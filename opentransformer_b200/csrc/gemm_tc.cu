// tcgen05 GEMM for sm_100a:  C[M,N] = A[M,K] * W[N,K]^T  (bf16 operands, fp32 accumulate in TMEM)
// with the fused epilogues the speech-transformer hot path needs (bias / ReLU / GLU / x*sqrt(d)+PE /
// residual / residual+LayerNorm / swish / gelu / tanh) and an implicit-GEMM mode for the 3x3 stride-2
// Conv2d subsampling layer (A gathered by a 5-D TMA tensor map, one 64-channel tap per k-block).
//
// Replaces the cuBLAS/oneDNN calls behind nn.Linear / nn.Conv2d at
//   otrans/module/attention.py:68,128-129,44   otrans/module/ffn.py:39-41
//   otrans/frontend/conv.py:63-64,146          otrans/decoder/transformer.py:181
//
// Structure (persistent, one CTA per SM, 640 threads):
//   warp 0 lane 0 : TMA producer   (A tile 128x64, B tile BNx64 per k-block, SWIZZLE_128B)
//   warp 1 lane 0 : tcgen05.mma issuer (UMMA 128 x BN x 16, 4 per k-block), tcgen05.commit -> mbarriers
//   warp 2        : TMEM allocator (2 accumulator stages x BN columns)
//   warps 4..19   : epilogue, four warpgroups: warp w reads TMEM lanes 32*(w%4).., warpgroup (w-4)/4 takes
//                   one quarter of the tile's columns.  tcgen05.ld -> registers -> fused math (bias / LN
//                   parameters broadcast from smem) -> staged in smem -> coalesced 16-byte global stores
//                   (one full output row segment per warp instruction; the residual tile is fetched the
//                   same way).  Round-1 profile: per-thread row stores were 32 sectors/request and the
//                   epilogue, not the MMA, bounded every GEMM (profiles/r1_*).
// Residual + LayerNorm epilogue (N = d_model <= 256): the output row is split over a thread-block CLUSTER
// of N/64 CTAs (64 columns each); per-row partial (sum, sum of squares) are exchanged through distributed
// shared memory (st.shared::cluster + remote mbarrier arrive), so the LN-fused GEMMs run on 4x more SMs
// than a one-CTA-per-row-block tiling would (63 -> 252 CTAs at cfg 2, 3 -> 12 in the decode loop).
// Three pipelines: smem full/empty ring (TMA <-> MMA), TMEM full/empty (MMA <-> epilogue), static
// round-robin tile scheduler, so the epilogue of tile i overlaps the MMAs of tile i+1.
#include <stdlib.h>
#include <string.h>

#include "dropout.cuh"
#include "launch.cuh"
#include "otb_internal.h"
#include "ptx.cuh"

namespace otb {

int g_tile_policy = 0;   // otb_set_tile_policy: 0 = lowest latency of a lone launch, 1 = least SM-time (concurrent batches)
unsigned long long* g_gemm_dbg = nullptr;
int g_gemm_dbg_mode = 0;
#define DBG_STAMP(i) do { if (p.dbg) p.dbg[blockIdx.x * 8 + (i)] = clock64(); } while (0)
// per-k-block traces of the first tile: kind 0 = TMA issue, 1 = full barrier observed by the MMA thread
#define DBG_KB(kind, kb) do { if (p.dbg && (kb) < 64) p.dbg[148 * 8 + (blockIdx.x * 2 + (kind)) * 64 + (kb)] = clock64(); } while (0)

// epilogue sub-phase stamps of the SECOND tile of every CTA (steady state): [148*8 + 148*2*64 + cta*16 + i]
#define DBG_EPI(i) do { if (p.dbg && it == 1 && et == 0) p.dbg[148 * 8 + 148 * 2 * 64 + blockIdx.x * 16 + (i)] = clock64(); } while (0)

static constexpr int BM = 128;
static constexpr int BK = 64;
static constexpr int kThreads = 640;
static constexpr int kEpiThreads = 512;
static constexpr int STG_PITCH_MAX = 512 + 16;          // bytes per staged row (+16 B pad: conflict-free 16 B accesses)
static constexpr int STG_BYTES = BM * STG_PITCH_MAX;    // 67,584
static constexpr int AUX_BYTES = 6144 + 8192;           // barriers, TMEM slot, bias / gamma / beta, row map | LN stats (wide tiles)

template <int BN>
struct GemmCfg {
    static constexpr int A_BYTES = BM * BK * 2;
    static constexpr int B_BYTES = BN * BK * 2;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int STAGES = (BN == 256) ? 3 : (BN == 128 ? 4 : 6);
    static constexpr int TMEM_COLS = 2 * BN;  // power of two for BN in {64,128,256}
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + STG_BYTES + AUX_BYTES + 1024;
};

// sigmoid(x) = 0.5 * tanh(x / 2) + 0.5 with ONE MUFU op (tanh.approx, |rel err| ~ 2^-11, far below the bf16 output
// rounding) instead of ex2 + rcp: the GLU epilogue of the K = 256 GEMMs is MUFU-bound (32 K sigmoids per 128x128 tile).
__device__ __forceinline__ float fast_sigmoid(float x) {
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.5f * x));
    return fmaf(0.5f, t, 0.5f);
}

__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, 512;" ::: "memory"); }

// 16 fp32 values -> staged row (bf16 or f32), 16-byte shared stores
__device__ __forceinline__ void stage16(uint8_t* row_ptr, int col, int out_f32, const float (&v)[16]) {
    if (out_f32) {
        float4* d = reinterpret_cast<float4*>(row_ptr + col * 4);
#pragma unroll
        for (int i = 0; i < 4; ++i) d[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
    } else {
        uint4* d = reinterpret_cast<uint4*>(row_ptr + col * 2);
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            uint4 u;
            u.x = pack_bf16(v[8 * i], v[8 * i + 1]);
            u.y = pack_bf16(v[8 * i + 2], v[8 * i + 3]);
            u.z = pack_bf16(v[8 * i + 4], v[8 * i + 5]);
            u.w = pack_bf16(v[8 * i + 6], v[8 * i + 7]);
            d[i] = u;
        }
    }
}

// TN = true: weight-gradient mode, C[M,N] = A^T B with A = dY [K rows, M cols] and B = X [K rows, N cols], both row-major,
// i.e. both operands are MN-major in shared memory (64x64 TMA boxes, LBO = 8 KB between 64-wide MN groups, SBO = 1 KB
// between 8-row K groups).  p.splitk > 1 splits the contraction over `splitk` tiles that accumulate with fp32 atomics.
template <int BN, int EPI, bool TN = false>
__global__ void __launch_bounds__(kThreads, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmParams p) {
    using Cfg = GemmCfg<BN>;
    constexpr int STAGES = Cfg::STAGES;
    constexpr int BN_OUT = (EPI == EPI_GLU) ? BN / 2 : BN;  // output columns per tile

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* stg = smem + STAGES * Cfg::STAGE_BYTES;
    uint8_t* aux = stg + STG_BYTES;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(aux);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tfull_bar = empty_bar + STAGES;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint64_t* ln_bar = tempty_bar + 2;                     // [2] cluster LayerNorm statistics exchange (alternate per tile)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(ln_bar + 2);
    float* s_bias = reinterpret_cast<float*>(aux + 256);   // [256]  (GLU: value half | gate half)
    float* s_gamma = s_bias + 256;                          // [256]
    float* s_beta = s_gamma + 256;                          // [256]
    int* s_rowmap = reinterpret_cast<int*>(s_beta + 256);   // [128] output row of each tile row, -1 = skip
    // LN partial statistics [2 tile parities][cluster ranks * 4 quarters <= 16][128 rows]: in the upper part of the
    // staging buffer when the LN tile is 64 wide (staging needs 128 x 144 B), else (one CTA per row block, at most
    // 4 partials per parity) in the pipeline-stage area's tail
    float2* s_stats = (BN == 64) ? reinterpret_cast<float2*>(stg + 32768)
                                 : (BN == 128 ? reinterpret_cast<float2*>(stg + 36864) : reinterpret_cast<float2*>(aux + 6144));   // BN 128: 2 x 8 x 128 partials = 16 KB above the 34 KB of staged rows
    const uint32_t cl_rank = (EPI == EPI_RESID_LN) ? cluster_ctarank() : 0;
    const uint32_t cl_size = (EPI == EPI_RESID_LN) ? cluster_nctarank() : 1;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    PDL_TRIGGER();   // the next kernel of the stream may be scheduled; it waits (griddepcontrol.wait) for this grid to finish
    if (threadIdx.x == 0) DBG_STAMP(0);

    const int m_tiles = p.conv ? (p.conv_B * p.conv_T1h + p.conv_R - 1) / p.conv_R : (p.M + BM - 1) / BM;
    const int n_tiles = (p.N + BN_OUT - 1) / BN_OUT;
    const int splitk = TN ? max(p.splitk, 1) : 1;
    const int num_tiles = m_tiles * n_tiles * splitk;
    const int num_kb_all = (p.K + BK - 1) / BK;
    // k-blocks of split ks: [ks*num_kb_all/splitk, (ks+1)*num_kb_all/splitk); without split-K: all of them
    auto kb_begin = [&](int tile) { return TN ? (int)(((long long)(tile % splitk) * num_kb_all) / splitk) : 0; };
    auto kb_end = [&](int tile) { return TN ? (int)(((long long)(tile % splitk + 1) * num_kb_all) / splitk) : num_kb_all; };
    const uint32_t a_tx = p.conv ? (uint32_t)(p.conv_R * p.conv_F2 * BK * 2) : (uint32_t)Cfg::A_BYTES;

    // One k-block load of the flat (tile, kb) sequence this CTA walks through.
    auto issue_load = [&](int tile, int kb, int stage) {
        const int mn = TN ? tile / splitk : tile;
        const int m_blk = mn / n_tiles, n_blk = mn % n_tiles;
        uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
        uint8_t* sb = sa + Cfg::A_BYTES;
        if (TN) {
            mbar_arrive_expect_tx(&full_bar[stage], (uint32_t)(Cfg::A_BYTES + Cfg::B_BYTES));
#pragma unroll
            for (int j = 0; j < BM / 64; ++j) tma_load_2d(sa + j * 8192, &tmA, &full_bar[stage], m_blk * BM + j * 64, kb * BK);
#pragma unroll
            for (int j = 0; j < BN / 64; ++j) tma_load_2d(sb + j * 8192, &tmB, &full_bar[stage], n_blk * BN + j * 64, kb * BK);
            return;
        }
        if (p.dbg_mode == 1) {  // profiling aid: signal "full" without moving any data
            mbar_arrive(&full_bar[stage]);
            return;
        }
        mbar_arrive_expect_tx(&full_bar[stage], a_tx + (uint32_t)Cfg::B_BYTES);
        if (p.conv) {
            // k-block -> (tap, channel chunk); tap (kh,kw): input row 2t'+kh, col 2f'+kw-1
            const int tap = kb / p.conv_cchunks, cc = kb % p.conv_cchunks;
            const int kh = tap / 3, kw = tap % 3;
            const int par_f = (kw == 1) ? 0 : 1, f0 = (kw == 0) ? -1 : 0;
            const int par_t = (kh == 1) ? 1 : 0, dt = (kh == 2) ? 1 : 0;
            tma_load_5d(sa, &tmA, &full_bar[stage], cc * BK, par_f, f0, par_t, m_blk * p.conv_R + dt);
        } else {
            tma_load_2d(sa, &tmA, &full_bar[stage], kb * BK, m_blk * BM);
        }
        if (EPI == EPI_GLU) {
            tma_load_2d(sb, &tmB, &full_bar[stage], kb * BK, n_blk * BN_OUT);
            tma_load_2d(sb + Cfg::B_BYTES / 2, &tmB, &full_bar[stage], kb * BK, p.N + n_blk * BN_OUT);
        } else {
            tma_load_2d(sb, &tmB, &full_bar[stage], kb * BK, n_blk * BN);
        }
    };

    // Producer state (meaningful in warp 0 lane 0 only): next load = (p_tile, p_kb) into p_stage.
    int p_tile = blockIdx.x, p_kb = kb_begin(blockIdx.x), p_stage = 0;
    uint32_t p_phase = 0;
    if (warp == 0) {
        if (lane == 0) {
            tma_prefetch_desc(&tmA);
            tma_prefetch_desc(&tmB);
            for (int i = 0; i < STAGES; ++i) {
                mbar_init(&full_bar[i], 1);
                mbar_init(&empty_bar[i], 1);
            }
            for (int i = 0; i < 2; ++i) {
                mbar_init(&tfull_bar[i], 1);
                mbar_init(&tempty_bar[i], kEpiThreads);
            }
            mbar_init(&ln_bar[0], 1);
            mbar_init(&ln_bar[1], 1);
            fence_barrier_init();
            PDL_WAIT();   // predecessor grid complete: its outputs (our A operand) may now be fetched
            // the first STAGES slots are free by construction: start the loads before the CTA-wide sync so
            // their latency overlaps the TMEM allocation
            for (int i = 0; i < STAGES && p_tile < num_tiles; ++i) {
                issue_load(p_tile, p_kb, p_stage);
                if (i == 0) DBG_STAMP(2);
                if (p_tile == (int)blockIdx.x) DBG_KB(0, p_kb);
                if (++p_kb >= kb_end(p_tile)) { p_tile += gridDim.x; p_kb = kb_begin(p_tile); }
                if (++p_stage == STAGES) { p_stage = 0; p_phase ^= 1; }
            }
        }
        __syncwarp();
    }
    if (warp == 2) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    PDL_WAIT();   // every thread, before its first global access (barrier init / TMEM allocation above overlap the predecessor)
    if (EPI == EPI_RESID_LN && cl_size > 1) cluster_sync_all();  // peers' mbarriers exist before any remote arrive
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (threadIdx.x == 0) DBG_STAMP(1);

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer (lane 0)
        if (lane == 0) {
            while (p_tile < num_tiles) {
                mbar_wait(&empty_bar[p_stage], p_phase ^ 1);
                issue_load(p_tile, p_kb, p_stage);
                if (p_tile == (int)blockIdx.x) DBG_KB(0, p_kb);
                if (++p_kb >= kb_end(p_tile)) { p_tile += gridDim.x; p_kb = kb_begin(p_tile); }
                if (++p_stage == STAGES) { p_stage = 0; p_phase ^= 1; }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer (lane 0)
        constexpr uint32_t idesc = umma_idesc_bf16(BN, TN, 128, TN);
        if (lane == 0) {
        int stage = 0;
        uint32_t phase = 0;
        int it = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
            const int as = it & 1;
            const uint32_t aph = (it >> 1) & 1;
            mbar_wait(&tempty_bar[as], aph ^ 1);
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)(as * BN);
            const int kb0 = kb_begin(tile), kb1 = kb_end(tile);
            for (int kb = kb0; kb < kb1; ++kb) {
                mbar_wait(&full_bar[stage], phase);
                tc_fence_after();
                if (it == 0 && kb == kb0) DBG_STAMP(3);
                if (it == 0) DBG_KB(1, kb);
                const uint32_t a_addr = smem_u32(smem + stage * Cfg::STAGE_BYTES);
                const uint32_t b_addr = a_addr + Cfg::A_BYTES;
                if (p.dbg_mode != 2) {
#pragma unroll
                    for (int k = 0; k < BK / 16; ++k) {
                        if (TN)   // MN-major operands: one k16 step = 16 rows of 128 B
                            umma_bf16(d_tmem, umma_desc_sw128(a_addr + k * 2048, 1024, 8192),
                                      umma_desc_sw128(b_addr + k * 2048, 1024, 8192), idesc, (uint32_t)(((kb - kb0) | k) != 0));
                        else
                            umma_bf16(d_tmem, umma_desc_sw128(a_addr + k * 32), umma_desc_sw128(b_addr + k * 32), idesc,
                                      (uint32_t)((kb | k) != 0));
                    }
                }
                umma_commit(&empty_bar[stage]);  // frees the smem slot once these MMAs have read it
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
            umma_commit(&tfull_bar[as]);  // accumulator complete -> epilogue
            if (it == 0) DBG_STAMP(4);
        }
        }
        __syncwarp();
    } else if (warp >= 4) {
        // ------------------------------------------------------------------ epilogue (512 threads, 16 warps)
        // warp w reads TMEM lanes 32*(w%4)..; the four warpgroups split the tile's columns into quarters and
        // walk them in 16-column chunks (4 warps per SM sub-partition hide the TMEM / MUFU / LDS latencies
        // that bounded the 8-warp version, profiles/r1_gemm_phases_v2.txt).
        const int et = threadIdx.x - 128;       // 0..511
        const int ewarp = warp - 4;             // 0..15
        const int quad = ewarp & 3;             // TMEM lane quadrant == warp % 4
        const int part = ewarp >> 2;            // column quarter handled by this warpgroup
        const int row_in_tile = quad * 32 + lane;
        const int esize = p.out_f32 ? 4 : 2;
        const int pitch = BN_OUT * esize + 16;
        uint8_t* my_row = stg + row_in_tile * pitch;
        constexpr int PART = BN_OUT / 4;        // output columns per warpgroup (16, 32 or 64)

        if (EPI == EPI_RESID_LN) {  // this CTA's 64-column slice of the LayerNorm affine parameters
            for (int i = et; i < BN; i += kEpiThreads) {
                s_gamma[i] = p.gamma[cl_rank * BN + i];
                s_beta[i] = p.beta[cl_rank * BN + i];
            }
        }
        int it = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
            const int mn_ = TN ? tile / splitk : tile;
            const int m_blk = mn_ / n_tiles, n_blk = mn_ % n_tiles;
            const int as = it & 1;
            const uint32_t aph = (it >> 1) & 1;
            const int col_base = n_blk * BN_OUT;             // first output column of the tile
            const int ncols = min(BN_OUT, p.N - col_base);   // valid output columns
            DBG_EPI(0);

            // ---- (a) per-tile smem setup: bias slice, row map, residual tile (all coalesced, loads batched)
            if (et < BN) {
                const int i = et;
                int c;
                if (EPI == EPI_GLU) c = (i < BN_OUT) ? col_base + i : p.N + col_base + (i - BN_OUT);
                else c = col_base + i;
                const bool ok = (EPI == EPI_GLU) ? ((i % BN_OUT) < ncols) : (i < ncols);
                s_bias[i] = (p.bias != nullptr && ok) ? p.bias[c] : 0.f;
            } else if (et >= 256 && et < 256 + BM) {
                const int rr = et - 256;
                int out_row;
                bool ok;
                if (p.conv) {
                    const int r = rr / p.conv_F2, f = rr % p.conv_F2;
                    const int bt = m_blk * p.conv_R + r;
                    const int b = bt / p.conv_T1h, t = bt % p.conv_T1h;
                    ok = (r < p.conv_R) && (b < p.conv_B) && (t < p.conv_T2);
                    out_row = (b * p.conv_T2 + t) * p.conv_F2 + f;
                } else {
                    out_row = m_blk * BM + rr;
                    ok = out_row < p.M;
                }
                s_rowmap[rr] = ok ? out_row : -1;
            }
            if (EPI == EPI_RESID || EPI == EPI_RESID_LN) {
                // residual rows are contiguous (no conv mode); 16-byte chunks, up to 8 independent loads per thread
                if ((ncols & 7) == 0) {
                    const int cpr = ncols >> 3;                        // 16-byte chunks per row
                    const int rows_here = min(BM, p.M - m_blk * BM);
                    const int total = rows_here * cpr;
                    const bf16* rbase = p.resid + (size_t)(m_blk * BM) * p.ldr + col_base;
                    for (int q0 = et; q0 < total; q0 += kEpiThreads * 8) {
                        uint4 tmp[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const int q = q0 + j * kEpiThreads;
                            if (q < total) tmp[j] = *reinterpret_cast<const uint4*>(rbase + (size_t)(q / cpr) * p.ldr + (q % cpr) * 8);
                        }
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const int q = q0 + j * kEpiThreads;
                            if (q < total) *reinterpret_cast<uint4*>(stg + (q / cpr) * pitch + (q % cpr) * 16) = tmp[j];
                        }
                    }
                } else {
                    for (int r = ewarp; r < BM; r += 16) {
                        const int grow = m_blk * BM + r;
                        if (grow >= p.M) continue;
                        const bf16* src = p.resid + (size_t)grow * p.ldr + col_base;
                        for (int c = lane; c < ncols; c += 32) reinterpret_cast<bf16*>(stg + r * pitch)[c] = src[c];
                    }
                }
            }
            epi_bar();
            DBG_EPI(1);

            // row validity / padding mask of this thread's row
            const int out_row = s_rowmap[row_in_tile];
            bool row_live = true;
            if (p.row_len != nullptr && out_row >= 0) {
                const int b = out_row / p.row_period, t = out_row % p.row_period;
                row_live = t < p.row_len[b];
            }

            mbar_wait(&tfull_bar[as], aph);
            tc_fence_after();
            if (it == 0 && et == 0) DBG_STAMP(5);
            DBG_EPI(2);
            const uint32_t t_row = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(as * BN);

            if (EPI == EPI_RESID_LN) {
                // Each thread owns PART = BN/4 columns of its row (16-column chunks).  Pass 1: v = resid + acc + bias,
                // (sum, sum of squares); v is parked back in TMEM when it does not fit one chunk.  The partials of
                // the 4 column quarters x cl_size CTAs meet through (distributed) shared memory.  Pass 2 normalises.
                float v[16];
                float s1 = 0.f, s2 = 0.f;
#pragma unroll 1
                for (int c = part * PART; c < (part + 1) * PART; c += 16) {
                    uint32_t r[16];
                    tmem_ld16(t_row + c, r);
                    tmem_ld_wait();
                    const uint4* rs = reinterpret_cast<const uint4*>(my_row + c * 2);
                    const float4* bs = reinterpret_cast<const float4*>(s_bias + c);
#pragma unroll
                    for (int i = 0; i < 2; ++i) {
                        const uint4 u = rs[i];
                        const float4 b0 = bs[2 * i], b1 = bs[2 * i + 1];
                        const float2 f0 = unpack_bf16(u.x), f1 = unpack_bf16(u.y), f2 = unpack_bf16(u.z), f3 = unpack_bf16(u.w);
                        const float rr[8] = {f0.x, f0.y, f1.x, f1.y, f2.x, f2.y, f3.x, f3.y};
                        const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            float x = __uint_as_float(r[8 * i + j]) + bb[j];
                            x = (row_live ? x : 0.f) + rr[j];
                            v[8 * i + j] = x;
                            s1 += x;
                            s2 += x * x;
                            r[8 * i + j] = __float_as_uint(x);
                        }
                    }
                    if (PART > 16) tmem_st16(t_row + c, r);
                }
                if (PART > 16) tmem_st_wait();
                if (PART == 16) {
                    tc_fence_before();
                    mbar_arrive(&tempty_bar[as]);  // accumulator consumed: the next tile's MMAs may start
                }
                // Tiles alternate between two (stats buffer, mbarrier) pairs: a peer that runs ahead signals the
                // OTHER barrier, so statistics of consecutive tiles can never be mixed.  Each remote store carries
                // its own byte count (st.async ... complete_tx), the owner expects 8 B x 512 threads x cl_size.
                const int par = it & 1;
                const int nslot = 4 * (int)cl_size;
                float2* my_slot = &s_stats[(par * nslot + (int)cl_rank * 4 + part) * BM + row_in_tile];
                if (cl_size == 1) {
                    *my_slot = make_float2(s1, s2);     // whole row in this CTA: plain shared memory + named barrier
                    epi_bar();
                } else {
                    if (et == 0) mbar_arrive_expect_tx(&ln_bar[par], (uint32_t)(8 * kEpiThreads) * cl_size);
                    const uint32_t slot = smem_u32(my_slot);
                    const uint32_t bar_local = smem_u32(&ln_bar[par]);
                    for (uint32_t dst = 0; dst < cl_size; ++dst)
                        st_async_f32x2(mapa_shared(slot, dst), s1, s2, mapa_shared(bar_local, dst));
                    mbar_wait_cluster(&ln_bar[par], (uint32_t)((it >> 1) & 1));
                }
                float t1 = 0.f, t2 = 0.f;
                for (int j = 0; j < 4 * (int)cl_size; ++j) {
                    const float2 o = s_stats[(par * nslot + j) * BM + row_in_tile];
                    t1 += o.x;
                    t2 += o.y;
                }
                const float inv_n = 1.0f / (float)(BN * cl_size);
                const float mean = t1 * inv_n;
                const float var = fmaxf(t2 * inv_n - mean * mean, 0.f);
                const float rstd = rsqrtf(var + p.eps);
#pragma unroll 1
                for (int c = part * PART; c < (part + 1) * PART; c += 16) {
                    if (PART > 16) {
                        uint32_t r[16];
                        tmem_ld16(t_row + c, r);
                        tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
                    }
                    const float4* gs = reinterpret_cast<const float4*>(s_gamma + c);
                    const float4* es = reinterpret_cast<const float4*>(s_beta + c);
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float4 g = gs[i], e = es[i];
                        v[4 * i] = (v[4 * i] - mean) * rstd * g.x + e.x;
                        v[4 * i + 1] = (v[4 * i + 1] - mean) * rstd * g.y + e.y;
                        v[4 * i + 2] = (v[4 * i + 2] - mean) * rstd * g.z + e.z;
                        v[4 * i + 3] = (v[4 * i + 3] - mean) * rstd * g.w + e.w;
                    }
                    stage16(my_row, c, 0, v);
                }
                if (PART > 16) {
                    tc_fence_before();
                    mbar_arrive(&tempty_bar[as]);
                }
            } else if (EPI == EPI_GLU) {
#pragma unroll 1
                for (int c = part * PART; c < (part + 1) * PART; c += 16) {
                    uint32_t ra[16], rg[16];
                    tmem_ld16(t_row + c, ra);
                    tmem_ld16(t_row + BN_OUT + c, rg);
                    tmem_ld_wait();
                    float v[16];
                    const float4* ba = reinterpret_cast<const float4*>(s_bias + c);
                    const float4* bg = reinterpret_cast<const float4*>(s_bias + BN_OUT + c);
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float4 x = ba[i], y = bg[i];
                        const float av[4] = {x.x, x.y, x.z, x.w}, gv[4] = {y.x, y.y, y.z, y.w};
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const float a = __uint_as_float(ra[4 * i + j]) + av[j];
                            const float g = __uint_as_float(rg[4 * i + j]) + gv[j];
                            v[4 * i + j] = row_live ? a * fast_sigmoid(g) : 0.f;
                        }
                    }
                    stage16(my_row, c, p.out_f32, v);
                }
            } else {
#pragma unroll 1
                for (int c = part * PART; c < (part + 1) * PART; c += 16) {
                    uint32_t r[16];
                    tmem_ld16(t_row + c, r);
                    tmem_ld_wait();
                    if (c >= ncols) continue;  // warp-uniform
                    float v[16];
                    float res[16];
                    if (EPI == EPI_RESID) {
                        const uint4* rs = reinterpret_cast<const uint4*>(my_row + c * 2);
#pragma unroll
                        for (int i = 0; i < 2; ++i) {
                            const uint4 u = rs[i];
                            const float2 f0 = unpack_bf16(u.x), f1 = unpack_bf16(u.y), f2 = unpack_bf16(u.z),
                                         f3 = unpack_bf16(u.w);
                            res[8 * i] = f0.x; res[8 * i + 1] = f0.y; res[8 * i + 2] = f1.x; res[8 * i + 3] = f1.y;
                            res[8 * i + 4] = f2.x; res[8 * i + 5] = f2.y; res[8 * i + 6] = f3.x; res[8 * i + 7] = f3.y;
                        }
                    }
                    const float* trow = nullptr;
                    if (EPI == EPI_TABLE)
                        trow = p.table + (size_t)((out_row >= 0 ? out_row : 0) % p.period) * p.N + col_base + c;
                    const uint32_t dseed = (EPI == EPI_RESID && p.drop_seed != nullptr) ? *p.drop_seed : 0u;
                    float bv[16];
                    {
                        const float4* bs = reinterpret_cast<const float4*>(s_bias + c);
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const float4 b4 = bs[i];
                            bv[4 * i] = b4.x; bv[4 * i + 1] = b4.y; bv[4 * i + 2] = b4.z; bv[4 * i + 3] = b4.w;
                        }
                    }
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        float x = __uint_as_float(r[i]) + bv[i];
                        if (EPI == EPI_RELU) x = fmaxf(x, 0.f);
                        if (EPI == EPI_SWISH) x = x * fast_sigmoid(x);
                        if (EPI == EPI_GELU) x = 0.5f * x * (1.0f + erff(x * 0.70710678118654752f));
                        if (EPI == EPI_TANH) x = tanhf(x);
                        if (EPI == EPI_TABLE) x = x * p.alpha + ((c + i < ncols) ? __ldg(trow + i) : 0.f);
                        if (!row_live) x = 0.f;
                        if (EPI == EPI_RESID && p.drop_seed != nullptr)   // nn.Dropout on the sub-layer output (transformer.py:54,61)
                            x = drop_keep(dseed, p.drop_site, (uint32_t)out_row, (uint32_t)(col_base + c + i), p.drop_thresh) ? x * p.drop_scale : 0.f;
                        if (EPI == EPI_RESID) x = res[i] + p.alpha * x;
                        v[i] = x;
                    }
                    stage16(my_row, c, p.out_f32, v);
                }
            }
            DBG_EPI(3);
            if (EPI != EPI_RESID_LN) {
                tc_fence_before();
                mbar_arrive(&tempty_bar[as]);  // TMEM stage is free for the next tile's MMAs
            }
            epi_bar();
            DBG_EPI(4);

            // ---- (e) coalesced copy-out: consecutive threads write consecutive 16-byte chunks of a row
            const int row_bytes = ncols * esize;
            if ((row_bytes & 15) == 0) {
                const int cpr = row_bytes >> 4;
                const int total = BM * cpr;
                uint8_t* obase = reinterpret_cast<uint8_t*>(p.out) + (size_t)col_base * esize;
                const size_t ld_bytes = (size_t)p.ldc * esize;
                for (int q0 = et; q0 < total; q0 += kEpiThreads * 4) {
                    uint4 tmp[4];
                    int orow[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int q = q0 + j * kEpiThreads;
                        orow[j] = -1;
                        if (q < total) {
                            const int r = q / cpr;
                            orow[j] = s_rowmap[r];
                            tmp[j] = *reinterpret_cast<const uint4*>(stg + r * pitch + (q % cpr) * 16);
                        }
                    }
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int q = q0 + j * kEpiThreads;
                        if (orow[j] < 0) continue;
                        if (TN && (splitk > 1 || p.accum)) {   // partial sums meet in the fp32 output (pre-zeroed, or a running gradient)
                            float* dst = reinterpret_cast<float*>(obase + (size_t)orow[j] * ld_bytes + (q % cpr) * 16);
                            atomicAdd(dst, __uint_as_float(tmp[j].x));
                            atomicAdd(dst + 1, __uint_as_float(tmp[j].y));
                            atomicAdd(dst + 2, __uint_as_float(tmp[j].z));
                            atomicAdd(dst + 3, __uint_as_float(tmp[j].w));
                        } else {
                            *reinterpret_cast<uint4*>(obase + (size_t)orow[j] * ld_bytes + (q % cpr) * 16) = tmp[j];
                        }
                    }
                }
            } else {
                for (int r = ewarp; r < BM; r += 16) {
                    const int orow = s_rowmap[r];
                    if (orow < 0) continue;
                    const uint8_t* src = stg + r * pitch;
                    uint8_t* dst = reinterpret_cast<uint8_t*>(p.out) + ((size_t)orow * p.ldc + col_base) * esize;
                    for (int off = lane * 2; off < row_bytes; off += 64)
                        *reinterpret_cast<uint16_t*>(dst + off) = *reinterpret_cast<const uint16_t*>(src + off);
                }
            }
            DBG_EPI(5);
            epi_bar();  // staging / bias smem may be rewritten for the next tile
            DBG_EPI(6);
            if (it == 0 && et == 0) DBG_STAMP(6);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) DBG_STAMP(7);
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
    }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
    static PFN_encodeTiled fn = nullptr;
    if (fn) return fn;
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
        return nullptr;
    fn = reinterpret_cast<PFN_encodeTiled>(ptr);
    return fn;
}

const char* encode_tmap_2d(CUtensorMap* m, const void* base, uint64_t cols, uint64_t rows, uint64_t ld_elems,
                           uint32_t box_cols, uint32_t box_rows, int swizzle_bytes) {
    PFN_encodeTiled enc = get_encode();
    if (!enc) return "cuTensorMapEncodeTiled unavailable (no CUDA driver?)";
    if ((reinterpret_cast<uintptr_t>(base) & 15) || (ld_elems & 7)) return "TMA operand must be 16-byte aligned with ld % 8 == 0";
    if (swizzle_bytes != 128 && swizzle_bytes != 64) return "encode_tmap_2d: swizzle must be 128 or 64 bytes";
    if (box_cols * 2 > (uint32_t)swizzle_bytes) return "encode_tmap_2d: box row wider than the swizzle span";
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {ld_elems * 2};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? nullptr : "cuTensorMapEncodeTiled(2d) failed";
}

// fp32, no swizzle: box_cols consecutive floats (a multiple of 4) of box_rows consecutive rows land densely in shared memory
const char* encode_tmap_2d_f32(CUtensorMap* m, const void* base, uint64_t cols, uint64_t rows, uint64_t ld_elems,
                               uint32_t box_cols, uint32_t box_rows) {
    PFN_encodeTiled enc = get_encode();
    if (!enc) return "cuTensorMapEncodeTiled unavailable (no CUDA driver?)";
    if ((reinterpret_cast<uintptr_t>(base) & 15) || (ld_elems & 3) || (box_cols & 3) || box_cols > 256 || box_rows > 256)
        return "fp32 TMA operand must be 16-byte aligned with ld % 4 == 0 and a box of <= 256 x 256";
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {ld_elems * 4};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? nullptr : "cuTensorMapEncodeTiled(2d, fp32) failed";
}

// conv1 output buffer [B, 2*T1h, 2*F1h, C] bf16 viewed as (c, f-parity, f/2, t-parity, b*T1h + t/2)
const char* encode_tmap_conv5d(CUtensorMap* m, const void* base, int C, int F1h, int T1h_total, uint32_t boxF,
                               uint32_t boxR) {
    PFN_encodeTiled enc = get_encode();
    if (!enc) return "cuTensorMapEncodeTiled unavailable (no CUDA driver?)";
    cuuint64_t dims[5] = {(cuuint64_t)C, 2, (cuuint64_t)F1h, 2, (cuuint64_t)T1h_total};
    cuuint64_t strides[4] = {(cuuint64_t)C * 2, (cuuint64_t)C * 4, (cuuint64_t)F1h * 2 * C * 2,
                             (cuuint64_t)F1h * 2 * C * 4};
    cuuint32_t box[5] = {64, 1, boxF, 1, boxR};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? nullptr : "cuTensorMapEncodeTiled(5d) failed";
}

int num_sms() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

template <int BN, int EPI>
static const char* launch_inst(cudaStream_t st, const CUtensorMap& ta, const CUtensorMap& tb, const GemmParams& p,
                               int num_tiles) {
    using Cfg = GemmCfg<BN>;
    static bool attr_set = false;
    if (!attr_set) {
        if (cudaFuncSetAttribute(gemm_tc_kernel<BN, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 Cfg::SMEM_BYTES) != cudaSuccess)
            return "cudaFuncSetAttribute(max dynamic smem) failed";
        attr_set = true;
    }
    int grid = num_tiles < num_sms() ? num_tiles : num_sms();
    if (EPI == EPI_RESID_LN && p.N / BN > 1) {
        const int cl = p.N / BN;              // CTAs per cluster == n-tiles per row block
        grid = (grid / cl) * cl;              // whole clusters only (num_tiles is a multiple of cl)
        if (grid < cl) return "gemm: grid smaller than one cluster";
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = dim3(grid);
        cfg.blockDim = dim3(kThreads);
        cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
        cfg.stream = st;
        cudaLaunchAttribute attr[2];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = cl;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[1].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        // co-resident clusters (GPC boundaries strand a few SMs): never launch more than fit in one wave
        static int max_clusters[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        if (cl <= 8 && max_clusters[cl] == 0) {
            int n = 0;
            if (cudaOccupancyMaxActiveClusters(&n, gemm_tc_kernel<BN, EPI>, &cfg) != cudaSuccess || n < 1) n = num_sms() / cl / 2;
            max_clusters[cl] = n;
        }
        if (cl <= 8 && grid > max_clusters[cl] * cl) {
            grid = max_clusters[cl] * cl;
            cfg.gridDim = dim3(grid);
        }
        prefer_max_smem_carveout(gemm_tc_kernel<BN, EPI>);
        cfg.numAttrs = pdl_enabled() ? 2 : 1;     // (the occupancy query above ran with the cluster attribute only)
        cudaError_t e = cudaLaunchKernelEx(&cfg, gemm_tc_kernel<BN, EPI>, ta, tb, p);
        return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
    }
    cudaError_t e = launch_pdl(gemm_tc_kernel<BN, EPI>, dim3(grid), dim3(kThreads), Cfg::SMEM_BYTES, st, ta, tb, p);
    return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
}

template <int BN>
static const char* launch_bn(cudaStream_t st, const CUtensorMap& ta, const CUtensorMap& tb, const GemmParams& p,
                             int epi, int num_tiles) {
    switch (epi) {
        case EPI_BIAS: return launch_inst<BN, EPI_BIAS>(st, ta, tb, p, num_tiles);
        case EPI_RELU: return launch_inst<BN, EPI_RELU>(st, ta, tb, p, num_tiles);
        case EPI_GLU: return launch_inst<BN, EPI_GLU>(st, ta, tb, p, num_tiles);
        case EPI_TABLE: return launch_inst<BN, EPI_TABLE>(st, ta, tb, p, num_tiles);
        case EPI_RESID: return launch_inst<BN, EPI_RESID>(st, ta, tb, p, num_tiles);
        case EPI_RESID_LN: return launch_inst<BN, EPI_RESID_LN>(st, ta, tb, p, num_tiles);
        case EPI_SWISH: return launch_inst<BN, EPI_SWISH>(st, ta, tb, p, num_tiles);
        case EPI_GELU: return launch_inst<BN, EPI_GELU>(st, ta, tb, p, num_tiles);
        case EPI_TANH: return launch_inst<BN, EPI_TANH>(st, ta, tb, p, num_tiles);
    }
    return "unknown epilogue";
}

// Pick the N tile that wastes the fewest MMA cycles across the persistent grid.
static int choose_bn(int m_tiles, int n_cols, int epi, int out_f32) {
    // Decode regime (<= 4 row blocks, M = batch x beam rows): every launch lasts 8-20 us whatever its tiling
    // (profiles/r1_ncu_decode_gemms_summary.txt) and utterance batches run concurrently on other streams, whose aggregate
    // throughput is bound by the SM-time the launches occupy (sum of CTAs x duration = 137 us of the whole GPU per decode
    // step, profiles/r1_bench_history.md).  So small problems take the WIDEST tile: 2-4x fewer CTAs for +1-2 us of latency.
    // Measured (profiles/r1_bench_history.md): policy 1 raises 8-lane throughput by 10-15 % and lengthens a lone 60-step
    // decode from 31.5 to 40.9 ms; the serving layer picks the policy (otb_set_tile_policy), latency is the default.
    const bool decode = (m_tiles <= 4) && g_tile_policy == 1;
    if (epi == EPI_RESID_LN) {
        // A tcgen05.mma from shared memory costs ~160 cycles for any N <= 256 (profiles/r1_bench_history.md), so a
        // 256-wide tile does the same main loop as four 64-wide ones: with enough row blocks to occupy the SMs (or under
        // the throughput policy) keep the whole row in one CTA; a lone small problem (decode, M = 320) is split over a
        // cluster of N/64 CTAs with DSMEM statistics, which shortens its launch by 2-4 us.
        // OTB_LN_BN = 64 | 128 | 256 overrides the column tile of the large-M case (tuning aid: the row is then split over
        // a cluster of N / BN CTAs with DSMEM statistics; 63 -> 126 -> 252 CTAs at cfg 2)
        static const int forced = [] { const char* e = getenv("OTB_LN_BN"); return e ? atoi(e) : 0; }();
        if (forced == 64 || forced == 128 || forced == 256) {
            if (m_tiles >= 32 && forced <= n_cols && n_cols % forced == 0) return forced;
        }
        // measured at cfg 2 (63 row blocks, N = 256; tools/encoder_time.py): one CTA per row block 1.509 ms per encoder pass,
        // the row split over a cluster of two 128-wide CTAs (126 CTAs) 1.436 ms, over four 64-wide CTAs 1.592 ms.  The split
        // is NOT the default: its statistics are combined from per-CTA (sum, sum of squares) partials, and on the benchmark
        // batch the 1-best agreement with the bf16-policy oracle dropped from 31 to 29 of 32 utterances for 5 % of 1.4 ms.
        return (m_tiles >= 32 || decode) ? n_cols : 64;
    }
    const int sms = num_sms();
    int best = 0;
    double best_cost = 1e30;
    const int cands[3] = {256, 128, 64};
    for (int i = 0; i < 3; ++i) {
        const int bn = cands[i];
        const int bn_out = (epi == EPI_GLU) ? bn / 2 : bn;
        if (bn_out * (out_f32 ? 4 : 2) > 512) continue;  // staged row must fit the staging pitch
        if (bn_out < 64) continue;                       // each epilogue warpgroup needs >= 16 columns
        const int n_tiles = (n_cols + bn_out - 1) / bn_out;
        const long tiles = (long)m_tiles * n_tiles;
        const long waves = (tiles + sms - 1) / sms;
        // large problems: fewest MMA cycles across the persistent grid (+48: per-tile fixed overhead in "column" units);
        // decode regime: least SM-time (+200: the fixed ~8 us of a launch expressed in the same units)
        const double cost = decode ? (double)tiles * (bn + 200) : (double)waves * (bn + 48);
        if (cost < best_cost - 1e-9) { best_cost = cost; best = bn; }
    }
    return best;
}

const char* gemm_launch(cudaStream_t st, const void* A, int lda, const void* W, int ldw, int w_rows, int epi,
                        GemmParams p, const CUtensorMap* conv_map) {
    if (p.M <= 0 || p.N <= 0 || p.K <= 0) return "gemm: empty problem";
    p.dbg = g_gemm_dbg;
    p.dbg_mode = g_gemm_dbg_mode;
    if (p.K % 8) return "gemm: K must be a multiple of 8";
    if (p.ldc % (p.out_f32 ? 4 : 8)) return "gemm: ldc must keep rows 16-byte aligned (ldc % 8 == 0 for bf16, % 4 for f32)";
    if (reinterpret_cast<uintptr_t>(p.out) & 15) return "gemm: out must be 16-byte aligned";
    if ((epi == EPI_RESID || epi == EPI_RESID_LN) && ((p.ldr % 8) || (reinterpret_cast<uintptr_t>(p.resid) & 15)))
        return "gemm: residual must be 16-byte aligned with ldr % 8 == 0";
    const int m_tiles = p.conv ? (p.conv_B * p.conv_T1h + p.conv_R - 1) / p.conv_R : (p.M + BM - 1) / BM;
    if (epi == EPI_RESID_LN && !(p.N == 64 || p.N == 128 || p.N == 256))
        return "gemm: fused residual+LayerNorm epilogue needs N in {64,128,256}";
    if (epi == EPI_RESID_LN && p.out_f32) return "gemm: fused residual+LayerNorm epilogue writes bf16";
    const int bn = choose_bn(m_tiles, p.N, epi, p.out_f32);
    if (bn == 0) return "gemm: no tile configuration";
    const int bn_out = (epi == EPI_GLU) ? bn / 2 : bn;
    const int n_tiles = (p.N + bn_out - 1) / bn_out;
    const int num_tiles = m_tiles * n_tiles;

    CUtensorMap ta, tb;
    const char* err;
    if (p.conv) {
        if (!conv_map) return "gemm: conv mode needs a conv tensor map";
        ta = *conv_map;
    } else {
        if ((err = encode_tmap_2d(&ta, A, (uint64_t)p.K, (uint64_t)p.M, (uint64_t)lda, BK, BM))) return err;
    }
    const uint32_t box_rows = (epi == EPI_GLU) ? (uint32_t)(bn / 2) : (uint32_t)bn;
    if ((err = encode_tmap_2d(&tb, W, (uint64_t)p.K, (uint64_t)w_rows, (uint64_t)ldw, BK, box_rows))) return err;

    switch (bn) {
        case 256: return launch_bn<256>(st, ta, tb, p, epi, num_tiles);
        case 128: return launch_bn<128>(st, ta, tb, p, epi, num_tiles);
        case 64: return launch_bn<64>(st, ta, tb, p, epi, num_tiles);
    }
    return "gemm: bad tile";
}

// Weight gradient dW[Nw, Kw] (fp32) = dY[Mact, Nw]^T X[Mact, Kw]  (both bf16 row-major): TN mode of the kernel above.
// The contraction (Mact rows, thousands) is split over enough tiles to fill the SMs; splits meet through fp32 atomics,
// so `out` must be zero on entry when the returned split count is > 1 (the launcher zeroes it with a memset node).
const char* gemm_wgrad_launch(cudaStream_t st, const void* dY, int lddy, const void* X, int ldx, float* out, int ldc,
                              int Mact, int Nw, int Kw, int accumulate) {
    if (Mact <= 0 || Nw <= 0 || Kw <= 0) return "wgrad: empty problem";
    if ((lddy % 8) || (ldx % 8) || (ldc % 4) || (reinterpret_cast<uintptr_t>(out) & 15)) return "wgrad: operands must be 16-byte aligned (ld % 8 bf16, ldc % 4 f32)";
    GemmParams p;
    memset(&p, 0, sizeof(p));
    p.M = Nw; p.N = Kw; p.K = Mact;
    p.out = out; p.ldc = ldc; p.out_f32 = 1; p.alpha = 1.f;
    p.dbg = nullptr; p.dbg_mode = 0;
    const int bn = (Kw > 64) ? 128 : 64;
    const int m_tiles = (Nw + BM - 1) / BM, n_tiles = (Kw + bn - 1) / bn;
    const int num_kb = (Mact + BK - 1) / BK;
    int splitk = num_sms() / (m_tiles * n_tiles);
    if (splitk > num_kb / 4) splitk = num_kb / 4;      // at least 4 k-blocks per split
    if (splitk < 1) splitk = 1;
    p.splitk = splitk;
    p.accum = accumulate ? 1 : 0;      // out += dY^T X (gradient accumulation): no memset, every tile adds atomically
    if (splitk > 1 && !accumulate) {
        cudaError_t e = cudaMemset2DAsync(out, (size_t)ldc * 4, 0, (size_t)Kw * 4, (size_t)Nw, st);
        if (e != cudaSuccess) return cudaGetErrorString(e);
    }
    CUtensorMap ta, tb;
    const char* err;
    if ((err = encode_tmap_2d(&ta, dY, (uint64_t)Nw, (uint64_t)Mact, (uint64_t)lddy, 64, 64))) return err;
    if ((err = encode_tmap_2d(&tb, X, (uint64_t)Kw, (uint64_t)Mact, (uint64_t)ldx, 64, 64))) return err;
    const int num_tiles = m_tiles * n_tiles * splitk;
    const int grid = num_tiles < num_sms() ? num_tiles : num_sms();
    cudaError_t e;
    if (bn == 128) {
        using Cfg = GemmCfg<128>;
        static bool attr = false;
        if (!attr) {
            if (cudaFuncSetAttribute(gemm_tc_kernel<128, EPI_BIAS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES) != cudaSuccess)
                return "cudaFuncSetAttribute(wgrad) failed";
            attr = true;
        }
        e = launch_pdl(gemm_tc_kernel<128, EPI_BIAS, true>, dim3(grid), dim3(kThreads), Cfg::SMEM_BYTES, st, ta, tb, p);
    } else {
        using Cfg = GemmCfg<64>;
        static bool attr = false;
        if (!attr) {
            if (cudaFuncSetAttribute(gemm_tc_kernel<64, EPI_BIAS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES) != cudaSuccess)
                return "cudaFuncSetAttribute(wgrad) failed";
            attr = true;
        }
        e = launch_pdl(gemm_tc_kernel<64, EPI_BIAS, true>, dim3(grid), dim3(kThreads), Cfg::SMEM_BYTES, st, ta, tb, p);
    }
    return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
}

}  // namespace otb
