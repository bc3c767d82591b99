// Fused masked multi-head attention for sm_100a (d_k = HD in {64, 96}):  softmax(Q K^T / sqrt(d_k) + mask) V
// Both contractions run on tcgen05 tensor cores with the score tile and the output tile in TMEM;
// the key-padding mask comes from lengths[b] (masks are always contiguous prefixes, SURVEY.md 8a),
// the causal mask from row/column indices, so no [B,h,T,T] tensor is ever materialised.
//
// Replaces BasedAttention.compute_context + the QK^T matmul:
//   otrans/module/attention.py:80 (scores), :34 (masked_fill -inf), :36 (softmax), :37 (weights @ V),
//   :41 (merge heads).  The reference also returns the [B,h,T1,T2] weights; no caller reads them
//   (model/speech2text.py:50,54), so they are not produced here.
//
// One CTA = 128 query rows of one (batch, head); 128 threads, thread i owns query row i (TMEM lane i).
// Keys are consumed in blocks of 128 with an online softmax:
//   TMA: Q tile [128x64], K block [128x64] (K-major) and V block [128 keys x 64] (MN-major B operand)
//   S  = Q K^T      : 4 x UMMA 128x128x16  -> TMEM columns [0,128)
//   P  = exp2(S*c - m) as bf16 written to smem in the canonical K-major SWIZZLE_128B layout
//   O' = P V        : 8 x UMMA 128x64x16   -> TMEM columns [128,192), rescaled + accumulated in registers
//
// HD = 96 (the Conformer recipe: d_model 384, 4 heads) adds a second, 32-column SWIZZLE_64B box per operand
// tile next to the 64-column SWIZZLE_128B one, so every TMA box lies inside the head's own 96 columns:
//   S  += 2 more UMMA k-steps read from the Q/K 64-byte-swizzled boxes
//   O2' = P V2      : 8 x UMMA 128x32x16   -> TMEM columns [192,224) (one MMA cannot span two swizzle modes)
// Shared memory 3 x 24 KB + 32 KB (P) ~ 105 KB: two CTAs still fit an SM.
#include "launch.cuh"
#include "otb_internal.h"
#include "ptx.cuh"

namespace otb {

// bytes of one [128 x HD] operand tile: a 16 KB SWIZZLE_128B box (+ an 8 KB SWIZZLE_64B box at HD = 96)
template <int HD>
static constexpr int att_tile_bytes() { return HD * 256; }
template <int HD>
static constexpr int att_smem() { return att_tile_bytes<HD>() * 3 + 32768 + 128 + 1024; }

template <int HD>
struct AttnMaps { CUtensorMap q, k, v; };                  // 64-column SWIZZLE_128B boxes
template <>
struct AttnMaps<96> { CUtensorMap q, k, v, q2, k2, v2; };  // + 32-column SWIZZLE_64B boxes at column +64

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// TMA of one [128 rows x HD] tile of operand `which` (0 = Q, 1 = K, 2 = V) at (col, row); its bytes complete on `bar`
__device__ __forceinline__ void load_tile(uint8_t* dst, const AttnMaps<64>& tm, int which, uint64_t* bar, int col, int row) {
    mbar_arrive_expect_tx(bar, 16384);
    tma_load_2d(dst, which == 0 ? &tm.q : which == 1 ? &tm.k : &tm.v, bar, col, row);
}
__device__ __forceinline__ void load_tile(uint8_t* dst, const AttnMaps<96>& tm, int which, uint64_t* bar, int col, int row) {
    mbar_arrive_expect_tx(bar, 16384 + 8192);
    tma_load_2d(dst, which == 0 ? &tm.q : which == 1 ? &tm.k : &tm.v, bar, col, row);
    tma_load_2d(dst + 16384, which == 0 ? &tm.q2 : which == 1 ? &tm.k2 : &tm.v2, bar, col + 64, row);
}

template <int HD, bool HAS_BD>
__global__ void __launch_bounds__(128, 2)
attn_tc_kernel(const __grid_constant__ AttnMaps<HD> tm, const AttnParams p) {
    static_assert(HD == 64 || HD == 96, "head width");
    constexpr int TILE = att_tile_bytes<HD>();
    PDL_TRIGGER();
    PDL_WAIT();   // before the first global read (kv_len) -- launch latency and CTA scheduling still overlap the predecessor
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sQ = smem;          // each tile: [128 x 64] SWIZZLE_128B, then (HD = 96) [128 x 32] SWIZZLE_64B
    uint8_t* sK = smem + TILE;
    uint8_t* sV = smem + 2 * TILE;
    uint8_t* sP = smem + 3 * TILE;  // 2 k-blocks x [128 rows x 128 B]
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + 3 * TILE + 32768);  // q, k, v, s, o
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 5);

    const int tid = threadIdx.x, warp = tid >> 5;
    const int q0 = blockIdx.x * 128, h = blockIdx.y, b = blockIdx.z;
    const int kv_len = p.kv_len ? min(p.kv_len[b], p.Tk) : p.Tk;
    int kv_end = kv_len;
    if (p.causal) kv_end = min(kv_end, q0 + 128);
    const int nblk = (kv_end + 127) / 128;

    if (warp == 0) {
        if (tid == 0) {
            for (int i = 0; i < 5; ++i) mbar_init(&bar[i], 1);
            fence_barrier_init();
            tma_prefetch_desc(&tm.q);
            tma_prefetch_desc(&tm.k);
            tma_prefetch_desc(&tm.v);
            if constexpr (HD == 96) {
                tma_prefetch_desc(&tm.q2);
                tma_prefetch_desc(&tm.k2);
                tma_prefetch_desc(&tm.v2);
            }
            // Q and the first K/V block are requested before the TMEM allocation / CTA sync
            load_tile(sQ, tm, 0, &bar[0], p.q_col0 + h * HD, b * p.Tq + q0);
            if (nblk > 0) {
                load_tile(sK, tm, 1, &bar[1], p.k_col0 + h * HD, b * p.Tk);
                load_tile(sV, tm, 2, &bar[2], p.v_col0 + h * HD, b * p.Tk);
            }
        }
        __syncwarp();
        tmem_alloc(tmem_slot, 256);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t t_row = tmem_base + ((uint32_t)(warp * 32) << 16);

    const int qi = q0 + tid;  // query index inside the utterance
    float m_run = -INFINITY, l_run = 0.f;
    float acc[HD];
#pragma unroll
    for (int i = 0; i < HD; ++i) acc[i] = 0.f;

    constexpr uint32_t idesc_s = umma_idesc_bf16(128, false);
    constexpr uint32_t idesc_o = umma_idesc_bf16(64, true);
    constexpr uint32_t idesc_o2 = umma_idesc_bf16(32, true);

    for (int blk = 0; blk < nblk; ++blk) {
        const uint32_t ph = blk & 1;
        const int key0 = blk * 128;
        if (tid == 0) {
            if (blk == 0) mbar_wait(&bar[0], 0);
            mbar_wait(&bar[1], ph);
            tc_fence_after();
            const uint32_t qa = smem_u32(sQ), ka = smem_u32(sK);
#pragma unroll
            for (int k = 0; k < 4; ++k)
                umma_bf16(tmem_base, umma_desc_sw128(qa + k * 32), umma_desc_sw128(ka + k * 32), idesc_s, (uint32_t)(k != 0));
            if constexpr (HD == 96) {   // dims [64,96): 64-byte rows, 8-row groups 512 B apart
#pragma unroll
                for (int k = 0; k < 2; ++k)
                    umma_bf16(tmem_base, umma_desc_sw64(qa + 16384 + k * 32), umma_desc_sw64(ka + 16384 + k * 32), idesc_s, 1u);
            }
            umma_commit(&bar[3]);
        }
        __syncwarp();
        mbar_wait(&bar[3], ph);
        tc_fence_after();
        if (tid == 0 && blk + 1 < nblk)   // S = QK^T has consumed the K block: prefetch the next one
            load_tile(sK, tm, 1, &bar[1], p.k_col0 + h * HD, b * p.Tk + key0 + 128);
        __syncwarp();

        // ---- pass 1: row maximum of the visible raw scores (the positive scale is applied afterwards)
        const int lim = p.causal ? min(kv_len, qi + 1) : kv_len;  // keys [0, lim) are visible to this row
        const float* bd_row = nullptr;
        if (HAS_BD) {
            const int qc = min(qi, p.Tq - 1);
            bd_row = p.bd + (((size_t)h * p.B + b) * p.Tq + qc) * p.ldbd + (p.Tq - 1 - qc);
        }
        float m_blk = -INFINITY;
#pragma unroll 1
        for (int c = 0; c < 128; c += 32) {
            uint32_t r[32];
            tmem_ld32(t_row + c, r);
            tmem_ld_wait();
            const int k0 = key0 + c;
            if (k0 + 32 <= lim) {
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    float sv = __uint_as_float(r[i]);
                    if (HAS_BD) sv += bd_row[k0 + i];
                    m_blk = fmaxf(m_blk, sv);
                }
            } else if (k0 < lim) {
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    float sv = __uint_as_float(r[i]);
                    if (HAS_BD && k0 + i < lim) sv += bd_row[k0 + i];
                    m_blk = fmaxf(m_blk, (k0 + i < lim) ? sv : -INFINITY);
                }
            }
        }
        m_blk *= p.scale_log2;  // -inf stays -inf
        const float m_new = fmaxf(m_run, m_blk);
        const float m_use = (m_new == -INFINITY) ? 0.f : m_new;
        const float alpha = (m_run == -INFINITY) ? 0.f : ex2_approx(m_run - m_use);
        float l_blk = 0.f;
        // ---- pass 2: probabilities -> bf16 -> smem (K-major, 128B swizzle)
#pragma unroll 1
        for (int c = 0; c < 128; c += 32) {
            uint32_t r[32];
            tmem_ld32(t_row + c, r);
            tmem_ld_wait();
            float pv[32];
            const int k0 = key0 + c;
            if (k0 + 32 <= lim) {
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    float sv = __uint_as_float(r[i]);
                    if (HAS_BD) sv += bd_row[k0 + i];
                    pv[i] = ex2_approx(fmaf(sv, p.scale_log2, -m_use));
                    l_blk += pv[i];
                }
            } else {
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    float sv = __uint_as_float(r[i]);
                    if (HAS_BD && k0 + i < lim) sv += bd_row[k0 + i];
                    pv[i] = (k0 + i < lim) ? ex2_approx(fmaf(sv, p.scale_log2, -m_use)) : 0.f;
                    l_blk += pv[i];
                }
            }
            uint8_t* prow = sP + (c >> 6) * 16384 + tid * 128;
            const int chunk0 = (c & 63) >> 3;  // 16-byte chunk index inside the 128-byte row
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                uint4 u;
                u.x = pack_bf16(pv[8 * j], pv[8 * j + 1]);
                u.y = pack_bf16(pv[8 * j + 2], pv[8 * j + 3]);
                u.z = pack_bf16(pv[8 * j + 4], pv[8 * j + 5]);
                u.w = pack_bf16(pv[8 * j + 6], pv[8 * j + 7]);
                *reinterpret_cast<uint4*>(prow + (((chunk0 + j) ^ (tid & 7)) << 4)) = u;
            }
        }
        l_run = l_run * alpha + l_blk;
        m_run = m_new;
        fence_proxy_async_smem();  // P (generic-proxy stores) -> visible to the tensor core's async proxy
        tc_fence_before();
        __syncthreads();

        if (tid == 0) {
            mbar_wait(&bar[2], ph);
            tc_fence_after();
            const uint32_t pa = smem_u32(sP), va = smem_u32(sV);
#pragma unroll
            for (int kk = 0; kk < 8; ++kk)
                umma_bf16(tmem_base + 128, umma_desc_sw128(pa + (kk >> 2) * 16384 + (kk & 3) * 32),
                          umma_desc_sw128(va + kk * 2048), idesc_o, (uint32_t)(kk != 0));
            if constexpr (HD == 96) {   // output dims [64,96) from the 64-byte-swizzled V box (16 keys = 1024 B per k-step)
#pragma unroll
                for (int kk = 0; kk < 8; ++kk)
                    umma_bf16(tmem_base + 192, umma_desc_sw128(pa + (kk >> 2) * 16384 + (kk & 3) * 32),
                              umma_desc_sw64(va + 16384 + kk * 1024), idesc_o2, (uint32_t)(kk != 0));
            }
            umma_commit(&bar[4]);
        }
        __syncwarp();
        mbar_wait(&bar[4], ph);
        tc_fence_after();
        if (tid == 0 && blk + 1 < nblk)   // PV has consumed the V block: prefetch the next one
            load_tile(sV, tm, 2, &bar[2], p.v_col0 + h * HD, b * p.Tk + key0 + 128);
        __syncwarp();
#pragma unroll
        for (int c = 0; c < HD; c += 32) {   // O at TMEM columns [128, 128 + HD)
            uint32_t r[32];
            tmem_ld32(t_row + 128 + c, r);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) acc[c + i] = acc[c + i] * alpha + __uint_as_float(r[i]);
        }
        tc_fence_before();
        __syncthreads();  // S/O TMEM and K/V/P smem may now be overwritten by the next block
    }

    if (qi < p.Tq) {
        if (p.lse) p.lse[((size_t)b * p.H + h) * p.Tq + qi] = (l_run > 0.f) ? m_run + log2f(l_run) : INFINITY;
        const float inv = (l_run > 0.f) ? 1.0f / l_run : 0.f;
        bf16* o = p.out + (size_t)(b * p.Tq + qi) * p.ldo + h * HD;
        if (p.resid) {
            const bf16* rr = p.resid + (size_t)(b * p.Tq + qi) * p.ldr + h * HD;
#pragma unroll
            for (int i = 0; i < HD; i += 8) {
                const uint4 u = *reinterpret_cast<const uint4*>(rr + i);
                const float2 a = unpack_bf16(u.x), bb = unpack_bf16(u.y), c = unpack_bf16(u.z), e = unpack_bf16(u.w);
                acc[i] = acc[i] * inv + a.x; acc[i + 1] = acc[i + 1] * inv + a.y;
                acc[i + 2] = acc[i + 2] * inv + bb.x; acc[i + 3] = acc[i + 3] * inv + bb.y;
                acc[i + 4] = acc[i + 4] * inv + c.x; acc[i + 5] = acc[i + 5] * inv + c.y;
                acc[i + 6] = acc[i + 6] * inv + e.x; acc[i + 7] = acc[i + 7] * inv + e.y;
            }
        } else {
#pragma unroll
            for (int i = 0; i < HD; ++i) acc[i] *= inv;
        }
#pragma unroll
        for (int i = 0; i < HD; i += 8) {
            uint4 u;
            u.x = pack_bf16(acc[i], acc[i + 1]);
            u.y = pack_bf16(acc[i + 2], acc[i + 3]);
            u.z = pack_bf16(acc[i + 4], acc[i + 5]);
            u.w = pack_bf16(acc[i + 6], acc[i + 7]);
            *reinterpret_cast<uint4*>(o + i) = u;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 256);
    }
}

template <int HD>
static const char* attn_launch_hd(cudaStream_t st, const void* q, int ldq, int q_rows, const void* k, int ldk, int k_rows,
                                  const void* v, int ldv, const AttnParams& p) {
    AttnMaps<HD> tm;
    const char* err;
    if ((err = encode_tmap_2d(&tm.q, q, (uint64_t)ldq, (uint64_t)q_rows, (uint64_t)ldq, 64, 128))) return err;
    if ((err = encode_tmap_2d(&tm.k, k, (uint64_t)ldk, (uint64_t)k_rows, (uint64_t)ldk, 64, 128))) return err;
    if ((err = encode_tmap_2d(&tm.v, v, (uint64_t)ldv, (uint64_t)k_rows, (uint64_t)ldv, 64, 128))) return err;
    if constexpr (HD == 96) {
        if ((err = encode_tmap_2d(&tm.q2, q, (uint64_t)ldq, (uint64_t)q_rows, (uint64_t)ldq, 32, 128, 64))) return err;
        if ((err = encode_tmap_2d(&tm.k2, k, (uint64_t)ldk, (uint64_t)k_rows, (uint64_t)ldk, 32, 128, 64))) return err;
        if ((err = encode_tmap_2d(&tm.v2, v, (uint64_t)ldv, (uint64_t)k_rows, (uint64_t)ldv, 32, 128, 64))) return err;
    }
    constexpr int smem = att_smem<HD>();
    static bool attr_set = false;
    if (!attr_set) {
        if (cudaFuncSetAttribute(attn_tc_kernel<HD, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess ||
            cudaFuncSetAttribute(attn_tc_kernel<HD, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess)
            return "cudaFuncSetAttribute(attn smem) failed";
        attr_set = true;
    }
    dim3 grid((p.Tq + 127) / 128, p.H, p.B);
    cudaError_t e = p.bd ? launch_pdl(attn_tc_kernel<HD, true>, grid, dim3(128), smem, st, tm, p)
                         : launch_pdl(attn_tc_kernel<HD, false>, grid, dim3(128), smem, st, tm, p);
    return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
}

const char* attn_launch(cudaStream_t st, const void* q, int ldq, int q_rows, const void* k, int ldk, int k_rows,
                        const void* v, int ldv, const AttnParams& p, int head_dim) {
    if (p.B <= 0 || p.H <= 0 || p.Tq <= 0 || p.Tk <= 0) return "attention: empty problem";
    if (head_dim == 64) return attn_launch_hd<64>(st, q, ldq, q_rows, k, ldk, k_rows, v, ldv, p);
    if (head_dim == 96) return attn_launch_hd<96>(st, q, ldq, q_rows, k, ldk, k_rows, v, ldv, p);
    return "head_dim must be 64 or 96";
}

}  // namespace otb
