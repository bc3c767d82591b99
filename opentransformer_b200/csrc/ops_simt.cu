// HBM-bound / latency-bound kernels of the hot path (no tensor cores): coalesced, vectorised,
// warp-shuffle reductions.  Each kernel cites the reference lines it replaces.
#include <math.h>

#include "launch.cuh"
#include "otb_internal.h"
#include "ptx.cuh"

namespace otb {

// ------------------------------------------------------------------------------------------------
// conv1: Conv2d(1 -> C1, 3x3, stride 2, padding (0,1)) + ReLU      otrans/frontend/conv.py:63-64
// in : x f32 [B, T, F]
// out: bf16 NHWC [B, 2*T1h, 2*F1h, C1]; columns f >= F1 are written as zero (they are the right
//      frequency padding of conv2); rows t >= T1 are never read for valid outputs and left untouched.
// HBM-bound on the output write (82 MB at cfg 2).  One CTA = 24 consecutive output rows of one
// utterance: the 49 input rows are staged in smem once, each thread keeps the 3x3 filters + bias of
// its 8 channels in registers and walks over (row, f1) positions, one 16-byte store per position,
// fully coalesced along (f1, c).  (With 8 rows per CTA the 80 weight loads per thread outnumbered the
// stores 8:1 -- 65 us for 22 MB, profiles/r1_ncu_layer_v5_summary.txt.)
// ------------------------------------------------------------------------------------------------
static constexpr int CONV1_ROWS = 24;

__global__ void __launch_bounds__(256) conv1_relu_nhwc_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                              const float* __restrict__ bias, bf16* __restrict__ out,
                                                              int B, int T, int F, int T1, int F1, int T1pad,
                                                              int F1pad, int C1) {
    PDL_TRIGGER();
    PDL_WAIT();
    extern __shared__ float sx[];  // [2*CONV1_ROWS + 1][F + 2]  (one zero column each side)
    const int chunks = (T1 + CONV1_ROWS - 1) / CONV1_ROWS;
    const int b = blockIdx.x / chunks, t1_0 = (blockIdx.x % chunks) * CONV1_ROWS;
    const int nrows = min(CONV1_ROWS, T1 - t1_0);
    const int W2 = F + 2;
    const int in_rows = 2 * nrows + 1;
    for (int i = threadIdx.x; i < in_rows * W2; i += blockDim.x) {
        const int r = i / W2, f = i % W2 - 1;
        sx[i] = (f >= 0 && f < F) ? x[((size_t)b * T + 2 * t1_0 + r) * F + f] : 0.f;
    }
    const int cgs = C1 / 8;             // channel groups of 8
    const int ppp = blockDim.x / cgs;   // positions per pass
    const int cg = threadIdx.x % cgs, pos0 = threadIdx.x / cgs;
    float wr[9][8], br[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        br[j] = bias[cg * 8 + j];
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) wr[tap][j] = w[(cg * 8 + j) * 9 + tap];
    }
    __syncthreads();
    if (pos0 >= ppp) return;
    const int npos = nrows * F1pad;
    for (int pos = pos0; pos < npos; pos += ppp) {
        const int r = pos / F1pad, f1 = pos % F1pad;
        float v[8];
        if (f1 < F1) {
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = br[j];
#pragma unroll
            for (int kh = 0; kh < 3; ++kh)
#pragma unroll
                for (int kw = 0; kw < 3; ++kw) {
                    const float xv = sx[(2 * r + kh) * W2 + 2 * f1 + kw];  // input col 2*f1 + kw - 1, +1 for the halo
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[j] = fmaf(xv, wr[kh * 3 + kw][j], v[j]);
                }
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = fmaxf(v[j], 0.f);
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = 0.f;
        }
        uint4 u;
        u.x = pack_bf16(v[0], v[1]);
        u.y = pack_bf16(v[2], v[3]);
        u.z = pack_bf16(v[4], v[5]);
        u.w = pack_bf16(v[6], v[7]);
        *reinterpret_cast<uint4*>(out + (((size_t)b * T1pad + t1_0 + r) * F1pad + f1) * C1 + cg * 8) = u;
    }
}

const char* conv1_launch(cudaStream_t st, const float* x, const float* w, const float* bias, bf16* out, int B, int T,
                         int F, int T1, int F1, int T1pad, int F1pad, int C1) {
    if (C1 % 8 || C1 > 2048) return "conv1: C1 must be a multiple of 8 (<= 2048)";
    size_t smem = (size_t)(2 * CONV1_ROWS + 1) * (F + 2) * sizeof(float);
    if (smem > 48 * 1024) return "conv1: F too large";
    const int chunks = (T1 + CONV1_ROWS - 1) / CONV1_ROWS;
    cudaError_t e = launch_pdl(conv1_relu_nhwc_kernel, dim3(B * chunks), dim3(256), smem, st, x, w, bias, out, B, T, F, T1, F1, T1pad,
                               F1pad, C1);
    return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
}

// ------------------------------------------------------------------------------------------------
// LayerNorm over the last dim (nn.LayerNorm, eps 1e-5): otrans/encoder/conformer.py:52,57,62,67,87,89
// bf16 in -> bf16 (or f32) out, fp32 statistics, warp per row, 16-byte loads.  An optional second
// affine LayerNorm is applied back to back (Conformer post_ffn_norm -> final_norm, conformer.py:87-89).
// ------------------------------------------------------------------------------------------------
template <int CH>  // CH = 16-byte chunks per lane (N = CH * 256)
__global__ void __launch_bounds__(256) layernorm_kernel(const bf16* __restrict__ x, int ldx, void* __restrict__ out,
                                                        int ldo, int out_f32, const float* __restrict__ g1,
                                                        const float* __restrict__ b1, const float* __restrict__ g2,
                                                        const float* __restrict__ b2, float eps, int M, int N) {
    PDL_TRIGGER();
    PDL_WAIT();
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= M) return;
    float v[CH * 8];
    const bf16* xr = x + (size_t)row * ldx;
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < CH; ++c) {
        const int col = (c * 32 + lane) * 8;
        if (col < N) {
            uint4 u = *reinterpret_cast<const uint4*>(xr + col);
            float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y), cc = unpack_bf16(u.z), d = unpack_bf16(u.w);
            v[c * 8 + 0] = a.x; v[c * 8 + 1] = a.y; v[c * 8 + 2] = b.x; v[c * 8 + 3] = b.y;
            v[c * 8 + 4] = cc.x; v[c * 8 + 5] = cc.y; v[c * 8 + 6] = d.x; v[c * 8 + 7] = d.y;
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) v[c * 8 + j] = 0.f;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) s += v[c * 8 + j];
    }
    for (int pass = 0; pass < 2; ++pass) {
        const float* g = pass ? g2 : g1;
        const float* bb = pass ? b2 : b1;
        if (pass == 1) {
            if (g2 == nullptr) break;
            s = 0.f;
#pragma unroll
            for (int i = 0; i < CH * 8; ++i) s += v[i];
        }
        const float mean = warp_sum(s) / N;
        float q = 0.f;
#pragma unroll
        for (int c = 0; c < CH; ++c) {
            const int col = (c * 32 + lane) * 8;
            if (col < N) {
#pragma unroll
                for (int j = 0; j < 8; ++j) { const float d = v[c * 8 + j] - mean; q += d * d; }
            }
        }
        const float rstd = rsqrtf(warp_sum(q) / N + eps);
#pragma unroll
        for (int c = 0; c < CH; ++c) {
            const int col = (c * 32 + lane) * 8;
            if (col < N) {
#pragma unroll
                for (int j = 0; j < 8; ++j) v[c * 8 + j] = (v[c * 8 + j] - mean) * rstd * g[col + j] + bb[col + j];
            }
        }
    }
#pragma unroll
    for (int c = 0; c < CH; ++c) {
        const int col = (c * 32 + lane) * 8;
        if (col < N) {
            if (out_f32) {
                float* o = reinterpret_cast<float*>(out) + (size_t)row * ldo + col;
                *reinterpret_cast<float4*>(o) = make_float4(v[c * 8], v[c * 8 + 1], v[c * 8 + 2], v[c * 8 + 3]);
                *reinterpret_cast<float4*>(o + 4) = make_float4(v[c * 8 + 4], v[c * 8 + 5], v[c * 8 + 6], v[c * 8 + 7]);
            } else {
                uint4 u;
                u.x = pack_bf16(v[c * 8], v[c * 8 + 1]);
                u.y = pack_bf16(v[c * 8 + 2], v[c * 8 + 3]);
                u.z = pack_bf16(v[c * 8 + 4], v[c * 8 + 5]);
                u.w = pack_bf16(v[c * 8 + 6], v[c * 8 + 7]);
                *reinterpret_cast<uint4*>(reinterpret_cast<bf16*>(out) + (size_t)row * ldo + col) = u;
            }
        }
    }
}

// N <= 256 fast path: one warp normalises 4 rows at a time so that 4 independent 16-byte loads (and 4
// independent reduction chains) are in flight per lane -- the one-row-per-warp version was latency-bound
// (14.8 us for 16 MB at Conformer cfg 4, profiles/r1_launches_conformer_v0.csv).
__global__ void __launch_bounds__(256) layernorm256_kernel(const bf16* __restrict__ x, int ldx, void* __restrict__ out,
                                                           int ldo, int out_f32, const float* __restrict__ g1,
                                                           const float* __restrict__ b1, const float* __restrict__ g2,
                                                           const float* __restrict__ b2, float eps, int M, int N) {
    PDL_TRIGGER();
    PDL_WAIT();
    constexpr int R = 4;
    const int lane = threadIdx.x & 31;
    const int row0 = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * R;
    if (row0 >= M) return;
    const int col = lane * 8;
    const bool live = col < N;
    float v[R][8];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        uint4 u = make_uint4(0, 0, 0, 0);
        if (live && row0 + r < M) u = *reinterpret_cast<const uint4*>(x + (size_t)(row0 + r) * ldx + col);
        const float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y), c = unpack_bf16(u.z), d = unpack_bf16(u.w);
        v[r][0] = a.x; v[r][1] = a.y; v[r][2] = b.x; v[r][3] = b.y; v[r][4] = c.x; v[r][5] = c.y; v[r][6] = d.x; v[r][7] = d.y;
    }
    float gg[8], bb[8];
    for (int pass = 0; pass < 2; ++pass) {
        const float* g = pass ? g2 : g1;
        const float* be = pass ? b2 : b1;
        if (g == nullptr) break;
#pragma unroll
        for (int j = 0; j < 8; ++j) { gg[j] = live ? g[col + j] : 0.f; bb[j] = live ? be[col + j] : 0.f; }
        float s[R], q[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            s[r] = 0.f;
#pragma unroll
            for (int j = 0; j < 8; ++j) s[r] += v[r][j];
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
#pragma unroll
            for (int r = 0; r < R; ++r) s[r] += __shfl_xor_sync(0xffffffffu, s[r], o);
#pragma unroll
        for (int r = 0; r < R; ++r) {
            s[r] /= N;
            q[r] = 0.f;
            if (live) {
#pragma unroll
                for (int j = 0; j < 8; ++j) { const float d = v[r][j] - s[r]; q[r] += d * d; }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
#pragma unroll
            for (int r = 0; r < R; ++r) q[r] += __shfl_xor_sync(0xffffffffu, q[r], o);
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const float rstd = rsqrtf(q[r] / N + eps);
#pragma unroll
            for (int j = 0; j < 8; ++j) v[r][j] = live ? (v[r][j] - s[r]) * rstd * gg[j] + bb[j] : 0.f;
        }
    }
    if (!live) return;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        if (row0 + r >= M) break;
        if (out_f32) {
            float* o = reinterpret_cast<float*>(out) + (size_t)(row0 + r) * ldo + col;
            *reinterpret_cast<float4*>(o) = make_float4(v[r][0], v[r][1], v[r][2], v[r][3]);
            *reinterpret_cast<float4*>(o + 4) = make_float4(v[r][4], v[r][5], v[r][6], v[r][7]);
        } else {
            uint4 u;
            u.x = pack_bf16(v[r][0], v[r][1]);
            u.y = pack_bf16(v[r][2], v[r][3]);
            u.z = pack_bf16(v[r][4], v[r][5]);
            u.w = pack_bf16(v[r][6], v[r][7]);
            *reinterpret_cast<uint4*>(reinterpret_cast<bf16*>(out) + (size_t)(row0 + r) * ldo + col) = u;
        }
    }
}

const char* layernorm_launch(cudaStream_t st, const bf16* x, int ldx, void* out, int ldo, int out_f32, const float* g1,
                             const float* b1, const float* g2, const float* b2, float eps, int M, int N) {
    if (N % 8 || ldx % 8 || N > 1024) return "layernorm: N must be a multiple of 8 and <= 1024";
    if ((out_f32 && ldo % 4) || (!out_f32 && ldo % 8)) return "layernorm: bad output stride";
    if (N <= 256) {
        const int rows_per_block = 8 * 4;
        cudaError_t e = launch_pdl(layernorm256_kernel, dim3((M + rows_per_block - 1) / rows_per_block), dim3(256), 0, st, x, ldx, out,
                                   ldo, out_f32, g1, b1, g2, b2, eps, M, N);
        return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
    }
    const int rows_per_block = 8;
    dim3 grid((M + rows_per_block - 1) / rows_per_block);
    const int ch = (N + 255) / 256;
    cudaError_t e;
    switch (ch) {
        case 1: e = launch_pdl(layernorm_kernel<1>, grid, dim3(256), 0, st, x, ldx, out, ldo, out_f32, g1, b1, g2, b2, eps, M, N); break;
        case 2: e = launch_pdl(layernorm_kernel<2>, grid, dim3(256), 0, st, x, ldx, out, ldo, out_f32, g1, b1, g2, b2, eps, M, N); break;
        case 3: e = launch_pdl(layernorm_kernel<3>, grid, dim3(256), 0, st, x, ldx, out, ldo, out_f32, g1, b1, g2, b2, eps, M, N); break;
        default: e = launch_pdl(layernorm_kernel<4>, grid, dim3(256), 0, st, x, ldx, out, ldo, out_f32, g1, b1, g2, b2, eps, M, N); break;
    }
    return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
}

// ------------------------------------------------------------------------------------------------
// Sinusoidal table: PE[p,2i] = sin(p*w_i), PE[p,2i+1] = cos(p*w_i), w_i = exp(-2i*ln(1e4)/d)
// otrans/module/pos.py:30-42 (recomputed on every call there; computed once per (first_pos, n, d) here)
// ------------------------------------------------------------------------------------------------
__global__ void sinusoid_table_kernel(float* __restrict__ out, int n_pos, int d, int first_pos) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pos * d) return;
    const int p = i / d + first_pos, c = i % d;
    const float w = expf((float)(c & ~1) * -(logf(10000.0f) / (float)d));
    const float a = (float)p * w;
    out[i] = (c & 1) ? cosf(a) : sinf(a);
}

const char* sinusoid_table_launch(cudaStream_t st, float* out, int n_pos, int d, int first_pos) {
    const int n = n_pos * d;
    sinusoid_table_kernel<<<(n + 255) / 256, 256, 0, st>>>(out, n_pos, d, first_pos);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
}

// ------------------------------------------------------------------------------------------------
// Embedding gather + positional encoding:  out[n] = emb[tok[n]] * sqrt(d) + PE[pos(n)]
// otrans/decoder/transformer.py:163,169  (+ module/pos.py:56)
// tok index:  tok[n * tok_stride + tok_off]; position: step_ptr ? *step_ptr : n % period
// ------------------------------------------------------------------------------------------------
__global__ void embed_posenc_kernel(const long long* __restrict__ tok, int tok_stride, const bf16* __restrict__ emb,
                                    const float* __restrict__ table, bf16* __restrict__ out, int N, int d, int period,
                                    const int* __restrict__ step_ptr, float xscale, int vocab) {
    PDL_TRIGGER();
    PDL_WAIT();
    const int n = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (n >= N) return;
    const int pos = step_ptr ? *step_ptr : (n % period);
    long long t = tok[(size_t)n * tok_stride];
    if (t < 0 || t >= vocab) t = 0;
    const bf16* e = emb + (size_t)t * d;
    const float* pe = table + (size_t)pos * d;
    for (int col = lane * 8; col < d; col += 256) {
        uint4 u = *reinterpret_cast<const uint4*>(e + col);
        float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y), c = unpack_bf16(u.z), dd = unpack_bf16(u.w);
        const float4 p0 = *reinterpret_cast<const float4*>(pe + col);
        const float4 p1 = *reinterpret_cast<const float4*>(pe + col + 4);
        uint4 o;
        o.x = pack_bf16(a.x * xscale + p0.x, a.y * xscale + p0.y);
        o.y = pack_bf16(b.x * xscale + p0.z, b.y * xscale + p0.w);
        o.z = pack_bf16(c.x * xscale + p1.x, c.y * xscale + p1.y);
        o.w = pack_bf16(dd.x * xscale + p1.z, dd.y * xscale + p1.w);
        *reinterpret_cast<uint4*>(out + (size_t)n * d + col) = o;
    }
}

const char* embed_posenc_launch(cudaStream_t st, const long long* tok, int tok_stride, const bf16* emb,
                                const float* table, bf16* out, int N, int d, int period, const int* step_ptr,
                                int vocab) {
    if (d % 8) return "embed: d must be a multiple of 8";
    cudaError_t e = launch_pdl(embed_posenc_kernel, dim3((N + 7) / 8), dim3(256), 0, st, tok, tok_stride, emb, table, out, N, d, period,
                               step_ptr, sqrtf((float)d), vocab);
    return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
}

// ------------------------------------------------------------------------------------------------
// Row log-softmax, fp32 (F.log_softmax of the last position's logits, decoder/transformer.py:206)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) log_softmax_kernel(const float* __restrict__ x, int ldx, float* __restrict__ out,
                                                          int ldo, int V) {
    PDL_TRIGGER();
    PDL_WAIT();
    __shared__ float red[8];
    __shared__ float bc;
    const float* xr = x + (size_t)blockIdx.x * ldx;
    float* orow = out + (size_t)blockIdx.x * ldo;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float m = -INFINITY;
    for (int i = threadIdx.x; i < V; i += 256) m = fmaxf(m, xr[i]);
    m = warp_max(m);
    if (lane == 0) red[warp] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = red[0];
        for (int i = 1; i < 8; ++i) t = fmaxf(t, red[i]);
        bc = t;
    }
    __syncthreads();
    m = bc;
    float s = 0.f;
    for (int i = threadIdx.x; i < V; i += 256) s += expf(xr[i] - m);
    s = warp_sum(s);
    __syncthreads();
    if (lane == 0) red[warp] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int i = 0; i < 8; ++i) t += red[i];
        bc = m + logf(t);
    }
    __syncthreads();
    const float lse = bc;
    for (int i = threadIdx.x; i < V; i += 256) orow[i] = xr[i] - lse;
}

const char* log_softmax_launch(cudaStream_t st, const float* x, int ldx, float* out, int ldo, int rows, int V) {
    cudaError_t e = launch_pdl(log_softmax_kernel, dim3(rows), dim3(256), 0, st, x, ldx, out, ldo, V);
    return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
}

// ------------------------------------------------------------------------------------------------
// Decode-time self-attention with a per-hypothesis KV cache (the `cache` the reference stubbed out,
// decoder/transformer.py:92-126,188-203).  One query (the newest token) per hypothesis; the prefix
// K/V of hypothesis n at position s' < step live in slot anc[n][s'] of step s' (beam reordering
// moves 4-byte ancestry entries, never K/V rows).  Warp = (hypothesis, head), d_k = HD in {64, 96};
// lane owns the bf16 pairs lane and lane + 32 (the latter only at HD = 96, lanes 0..15).
// Also appends the current K/V to the cache.
//   qkv   bf16 [N, 3d] (Q | K | V of the current token, attention.py:73 split order)
//   kc,vc bf16 [Lmax, N, d]
//   anc   int32 [2, N, Lmax]  (ping-pong, buffer (step & 1) is current)
// ------------------------------------------------------------------------------------------------
template <int HD>
__global__ void __launch_bounds__(128, HD == 64 ? 6 : 4) decode_self_attn_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ kc,
                                                               bf16* __restrict__ vc, const int* __restrict__ anc,
                                                               const int* __restrict__ step_ptr, bf16* __restrict__ out,
                                                               int N, int H, int Lmax, float scale, int keys_pad) {
    PDL_TRIGGER();
    PDL_WAIT();
    // Lanes run over KEYS: each lane owns up to KPL cached positions, resolves their slots through the
    // ancestry table and pulls the whole K and V rows (HD * 2 bytes) with 16-byte loads -- all loads of a lane are
    // independent, so the kernel costs ~3 dependent memory round trips (anc -> K/V -> out) instead of a
    // serial walk over the prefix.  V rows go through smem so that the P.V reduction is a column sum.
    constexpr int KPL = 4;               // keys per lane -> up to 128 cached positions
    constexpr int NC = HD / 8;           // 16-byte chunks per K/V row
    constexpr int NP = HD / 2;           // bf16 pairs per row
    // staged V row pitch in chunks: HD = 64 rotates the 8 chunks of row s by s; HD = 96 pads the 12 chunks to 13
    // (an odd pitch spreads the 8 rows of a store phase over all 8 bank groups)
    constexpr int PITCH = HD == 64 ? 8 : NC + 1;
    extern __shared__ uint4 sv_raw[];    // [warps][keys_pad][PITCH x 16 B]  V rows (bf16)
    const int n = blockIdx.x;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int nw = blockDim.x >> 5;
    const int d = H * HD;
    const int step = *step_ptr;
    const int nkeys = step + 1;
    const int* an = anc + ((size_t)(step & 1) * N + n) * Lmax;
    uint4* sv = sv_raw + (size_t)wib * keys_pad * PITCH;    // [keys_pad][PITCH x 16 B] per warp
    // q lives in shared memory (every lane needs all HD dims: HD registers per thread otherwise, which capped the kernel
    // at 3 resident CTAs per SM -- the SM-time of this latency-bound kernel is what concurrent batches compete for)
    float* sq = reinterpret_cast<float*>(sv_raw + (size_t)(blockDim.x >> 5) * keys_pad * PITCH) + wib * HD;
    auto v_word = [&](int s, int w) {    // 4-byte word w (dims 2w, 2w+1) of staged V row s
        const uint32_t* svw = reinterpret_cast<const uint32_t*>(sv);
        if constexpr (HD == 64) return svw[(s * 8 + (((w >> 2) + s) & 7)) * 4 + (w & 3)];   // chunks were rotated by s
        else return svw[s * PITCH * 4 + w];
    };
    for (int h = wib; h < H; h += nw) {
        const bf16* base = qkv + (size_t)n * 3 * d + h * HD;
        // append the newest K/V to the cache
        __syncwarp();
#pragma unroll
        for (int w = lane; w < NP; w += 32) {
            const uint32_t kcur = *reinterpret_cast<const uint32_t*>(base + d + 2 * w);
            const uint32_t vcur = *reinterpret_cast<const uint32_t*>(base + 2 * d + 2 * w);
            const size_t cur_off = ((size_t)step * N + n) * d + h * HD + 2 * w;
            *reinterpret_cast<uint32_t*>(kc + cur_off) = kcur;
            *reinterpret_cast<uint32_t*>(vc + cur_off) = vcur;
            const float2 qq = unpack_bf16(*reinterpret_cast<const uint32_t*>(base + 2 * w));
            sq[2 * w] = qq.x;
            sq[2 * w + 1] = qq.y;
        }
        __syncwarp();
        int slot[KPL];
#pragma unroll
        for (int j = 0; j < KPL; ++j) {
            const int s = lane + 32 * j;
            slot[j] = (s < step) ? an[s] : n;
        }
        float sc[KPL];
        float mx = -INFINITY;
#pragma unroll
        for (int j = 0; j < KPL; ++j) {
            const int s = lane + 32 * j;
            sc[j] = -INFINITY;
            if (s < nkeys) {   // warp-divergent only in the last group
                const bf16* krow = (s == step) ? base + d : kc + ((size_t)s * N + slot[j]) * d + h * HD;
                const bf16* vrow = (s == step) ? base + 2 * d : vc + ((size_t)s * N + slot[j]) * d + h * HD;
                uint4 ku[NC], vu[NC];
#pragma unroll
                for (int i = 0; i < NC; ++i) ku[i] = *reinterpret_cast<const uint4*>(krow + 8 * i);
#pragma unroll
                for (int i = 0; i < NC; ++i) vu[i] = *reinterpret_cast<const uint4*>(vrow + 8 * i);
                float dot = 0.f;
#pragma unroll
                for (int i = 0; i < NC; ++i) {
                    const float2 a = unpack_bf16(ku[i].x), b = unpack_bf16(ku[i].y), c = unpack_bf16(ku[i].z),
                                 e = unpack_bf16(ku[i].w);
                    const float4 q0 = *reinterpret_cast<const float4*>(sq + 8 * i);      // broadcast reads
                    const float4 q1 = *reinterpret_cast<const float4*>(sq + 8 * i + 4);
                    dot += q0.x * a.x + q0.y * a.y + q0.z * b.x + q0.w * b.y + q1.x * c.x + q1.y * c.y + q1.z * e.x + q1.w * e.y;
                }
                sc[j] = dot * scale;
                mx = fmaxf(mx, sc[j]);
#pragma unroll
                for (int i = 0; i < NC; ++i) {
                    if constexpr (HD == 64) sv[s * 8 + ((i + s) & 7)] = vu[i];   // rotate chunks: conflict-free rows
                    else sv[s * PITCH + i] = vu[i];
                }
            }
        }
        mx = warp_max(mx);
        float l = 0.f;
#pragma unroll
        for (int j = 0; j < KPL; ++j) {
            sc[j] = (lane + 32 * j < nkeys) ? __expf(sc[j] - mx) : 0.f;
            l += sc[j];
        }
        l = warp_sum(l);
        __syncwarp();
        // P.V as a column sum over the staged V rows: lane owns the bf16 pairs lane (+ lane + 32)
        constexpr int NW = (NP + 31) / 32;
        const bool second = NW > 1 && lane + 32 < NP;
        float ax[NW], ay[NW];
#pragma unroll
        for (int u = 0; u < NW; ++u) ax[u] = ay[u] = 0.f;
#pragma unroll
        for (int j = 0; j < KPL; ++j) {
            const int cnt = min(32, nkeys - 32 * j);
            if (cnt <= 0) break;   // warp-uniform
#pragma unroll 4
            for (int t = 0; t < cnt; ++t) {
                const int s = t + 32 * j;
                const float pw = __shfl_sync(0xffffffffu, sc[j], t);
                const float2 vf = unpack_bf16(v_word(s, lane));
                ax[0] = fmaf(pw, vf.x, ax[0]);
                ay[0] = fmaf(pw, vf.y, ay[0]);
                if constexpr (NW > 1) {
                    if (second) {
                        const float2 vg = unpack_bf16(v_word(s, lane + 32));
                        ax[NW - 1] = fmaf(pw, vg.x, ax[NW - 1]);
                        ay[NW - 1] = fmaf(pw, vg.y, ay[NW - 1]);
                    }
                }
            }
        }
        const float inv = 1.0f / l;
        bf16* orow = out + (size_t)n * d + h * HD;
        *reinterpret_cast<uint32_t*>(orow + 2 * lane) = pack_bf16(ax[0] * inv, ay[0] * inv);
        if constexpr (NW > 1) {
            if (second) *reinterpret_cast<uint32_t*>(orow + 2 * (lane + 32)) = pack_bf16(ax[NW - 1] * inv, ay[NW - 1] * inv);
        }
        __syncwarp();
    }
}

template <int HD>
static const char* decode_self_attn_launch_hd(cudaStream_t st, const bf16* qkv, bf16* kc, bf16* vc, const int* anc,
                                              const int* step_ptr, bf16* out, int N, int H, int Lmax) {
    const int warps = H < 4 ? H : 4;
    // V staging sized by the longest prefix this search can reach (not the 128-key maximum): at max_len 60 this halves the
    // shared memory per CTA and doubles the resident CTAs of this latency-bound kernel (less SM-time per decode step)
    constexpr int PITCH = HD == 64 ? 8 : HD / 8 + 1;
    constexpr int MAX_SMEM = 4 * 128 * PITCH * 16 + 4 * HD * (int)sizeof(float);
    const int keys_pad = (Lmax + 31) / 32 * 32;
    const size_t smem = (size_t)warps * keys_pad * PITCH * 16 + (size_t)warps * HD * sizeof(float);   // V rows | q per warp
    static bool attr_set = false;
    if (!attr_set) {
        if (cudaFuncSetAttribute(decode_self_attn_kernel<HD>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 MAX_SMEM > 80 * 1024 ? MAX_SMEM : 80 * 1024) != cudaSuccess)
            return "cudaFuncSetAttribute(decode_self_attn) failed";
        attr_set = true;
    }
    cudaError_t e = launch_pdl(decode_self_attn_kernel<HD>, dim3(N), dim3(warps * 32), smem, st, qkv, kc, vc, anc, step_ptr, out, N,
                               H, Lmax, HD == 64 ? 0.125f : 1.0f / sqrtf((float)HD), keys_pad);
    return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
}

const char* decode_self_attn_launch(cudaStream_t st, const bf16* qkv, bf16* kc, bf16* vc, const int* anc,
                                    const int* step_ptr, bf16* out, int N, int H, int Lmax, int head_dim) {
    if (Lmax > 128) return "decode_self_attn: at most 128 cached positions (max_len <= 128)";
    if (head_dim == 64) return decode_self_attn_launch_hd<64>(st, qkv, kc, vc, anc, step_ptr, out, N, H, Lmax);
    if (head_dim == 96) return decode_self_attn_launch_hd<96>(st, qkv, kc, vc, anc, step_ptr, out, N, H, Lmax);
    return "head_dim must be 64 or 96";
}

// ------------------------------------------------------------------------------------------------
// Stand-alone PositionalEncoding.forward: out = x * alpha + table[row % period]   (module/pos.py:56)
// (the fused path does this in the front-end Linear's epilogue; this kernel serves the module-level
// drop-in API where frontend and encoder are called separately).  x f32 or bf16 -> bf16.
// ------------------------------------------------------------------------------------------------
__global__ void scale_add_table_kernel(const void* __restrict__ x, int ldx, int x_f32, bf16* __restrict__ out, int ldo,
                                       float alpha, const float* __restrict__ table, int period, int M, int N) {
    PDL_TRIGGER();
    PDL_WAIT();
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int row = (int)(i / N), col = (int)(i % N);
    if (row >= M) return;
    const float v = x_f32 ? reinterpret_cast<const float*>(x)[(size_t)row * ldx + col]
                          : __bfloat162float(reinterpret_cast<const bf16*>(x)[(size_t)row * ldx + col]);
    const float t = table ? table[(size_t)(row % period) * N + col] : 0.f;
    out[(size_t)row * ldo + col] = __float2bfloat16(v * alpha + t);
}

const char* scale_add_table_launch(cudaStream_t st, const void* x, int ldx, int x_f32, bf16* out, int ldo, float alpha,
                                   const float* table, int period, int M, int N) {
    const size_t n = (size_t)M * N;
    cudaError_t e = launch_pdl(scale_add_table_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, st, x, ldx, x_f32, out, ldo, alpha,
                               table, period, M, N);
    return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
}

// ------------------------------------------------------------------------------------------------
// Conformer convolution-module middle: depthwise Conv1d over time (k taps, zero padding (k-1)/2) +
// eval-mode BatchNorm (folded into w/b by the caller) + swish.   otrans/module/conformer.py:48-52
// x, out bf16 [B*T, d].  HBM-bound: thread = (row, 8 channels), 16-byte loads of the k neighbour rows
// (re-reads hit L1/L2), fp32 math.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) dwconv_swish_kernel(const bf16* __restrict__ x, const float* __restrict__ w,
                                                           const float* __restrict__ b, bf16* __restrict__ out, int B,
                                                           int T, int d, int k) {
    PDL_TRIGGER();
    PDL_WAIT();
    const int cg = d / 8;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)B * T * cg) return;
    const int c0 = (int)(i % cg) * 8;
    const int row = (int)(i / cg);
    const int t = row % T;
    const int pad = (k - 1) / 2;
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = b[c0 + j];
    for (int tap = 0; tap < k; ++tap) {
        const int tt = t + tap - pad;
        if (tt < 0 || tt >= T) continue;
        const uint4 u = *reinterpret_cast<const uint4*>(x + (size_t)(row + tap - pad) * d + c0);
        const float2 a = unpack_bf16(u.x), bb = unpack_bf16(u.y), c = unpack_bf16(u.z), e = unpack_bf16(u.w);
        const float xv[8] = {a.x, a.y, bb.x, bb.y, c.x, c.y, e.x, e.y};
        const float4 w0 = *reinterpret_cast<const float4*>(w + (size_t)tap * d + c0);
        const float4 w1 = *reinterpret_cast<const float4*>(w + (size_t)tap * d + c0 + 4);
        const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = fmaf(xv[j], wv[j], acc[j]);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = acc[j] * __fdividef(1.0f, 1.0f + __expf(-acc[j]));
    uint4 o;
    o.x = pack_bf16(acc[0], acc[1]);
    o.y = pack_bf16(acc[2], acc[3]);
    o.z = pack_bf16(acc[4], acc[5]);
    o.w = pack_bf16(acc[6], acc[7]);
    *reinterpret_cast<uint4*>(out + (size_t)row * d + c0) = o;
}

const char* dwconv_swish_launch(cudaStream_t st, const bf16* x, const float* w, const float* b, bf16* out, int B, int T,
                                int d, int k) {
    if (d % 8 || !(k & 1)) return "dwconv: d must be a multiple of 8 and k odd";
    const size_t n = (size_t)B * T * (d / 8);
    cudaError_t e = launch_pdl(dwconv_swish_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, st, x, w, b, out, B, T, d, k);
    return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
}

}  // namespace otb
