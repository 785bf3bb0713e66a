// tcgen05 / TMEM spatial self-attention (attention.py:56-74), bf16 or fp16 (a template parameter, format from Fmt16),
// head_dim 32 / 64 / 128, any H x W with W <= 128.
// Tiles are R = floor(128 / W) whole image rows (<= 128 tokens); a tile may be ragged (R*W < 128) and the last one partial.
// Q, K, V (and dO) arrive by TMA straight out of the NHWC `qkv` tensor (4-D maps over (channel, x, y, image): the halo
// pixels are not in the box, the permute + contiguous copies of attention.py:63-65 never exist).
//
// Forward, one CTA per (image, head, query tile), a loop over key tiles (flash attention with an online softmax):
//   S_j = Q K_j^T  tcgen05.mma, M = 128 queries, N = the key tile padded to 16, K = head_dim; Q and K as 16-channel K-major
//                  chunks (SWIZZLE_32B); S double-buffered in tensor memory (columns 0 / 128) so S_{j+1} is computed while
//                  the softmax warps work on S_j; K / V double-buffered in shared memory
//   P_j            128 threads, one query row each: running max m and sum l, P_j = exp(S_j - m) as 16-bit K-major chunks
//   O += P_j V_j   B = V read MN-major (head_dim contiguous, 64-channel SWIZZLE_128B boxes; head_dim 128 = two boxes and two
//                  N = 64 halves) into TMEM columns 256..; the softmax threads fold it into fp32 registers,
//                  o = o * exp(m_old - m_new) + P_j V_j, and store o / l and lse = m * scale + log l.
// N <= 256 with head_dim <= 64 keeps one all-keys tile (the UNet's blocks: today's arithmetic).
//
// Attention is <0.4 % of the model FLOPs but 6 % of the CelebA256 step with the CUDA-core kernels of attn_kernels.cu
// (profiles/r2_launches_step_celeba256_summary.txt); those remain the fp32 path and the fallback for other head sizes
// and W > 128.
#include "common.cuh"
#include <cuda.h>
#include <cudaTypedefs.h>
#include <math.h>

extern int ddpm_encode_tiled16(CUtensorMap* m, CUtensorMapDataType type, void* base, int rank, const uint64_t* dims,
                               const uint64_t* strides_bytes, const uint32_t* box, int swizzle_bytes);      // conv_tc.cu

namespace {

#define ATC_THREADS 192          // warp 0: TMA, warp 1: MMA issue, warps 2..5: softmax + epilogue (one TMEM lane quarter each)

__device__ __forceinline__ uint32_t s32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mb_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(s32(bar)), "r"(count));
}
__device__ __forceinline__ void mb_expect(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(s32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mb_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(s32(bar)) : "memory");
}
__device__ __forceinline__ void mb_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "AW_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra AD_%=;\n\t"
        "bra AW_%=;\n\t"
        "AD_%=:\n\t}" ::"r"(s32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma4(void* dst, const CUtensorMap* m, uint64_t* bar, int c, int x, int y, int n) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
                 ::"r"(s32(dst)), "l"(m), "r"(s32(bar)), "r"(c), "r"(x), "r"(y), "r"(n) : "memory");
}
__device__ __forceinline__ void tm_alloc(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tm_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void mma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(s32(bar)) : "memory");
}
__device__ __forceinline__ void tm_ld16(uint32_t taddr, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr));
}
__device__ __forceinline__ void tm_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout): address, LBO, SBO in 16-byte units, version 1, layout type
__device__ __forceinline__ uint64_t mdesc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)(layout & 7) << 61;
    return d;
}
// instruction descriptors: 16-bit x 16-bit -> fp32, M = 128.  S-type: both operands K-major, N = n.  O-type: B MN-major, N = 64.
template <typename T> __device__ __forceinline__ uint32_t idesc_kk(int n) { return (1u << 4) | Fmt16<T>::idesc_ab | ((uint32_t)(n >> 3) << 17) | ((128u >> 4) << 24); }
template <typename T> __device__ __forceinline__ uint32_t idesc_mn64() { return (1u << 4) | Fmt16<T>::idesc_ab | (1u << 16) | ((64u >> 3) << 17) | ((128u >> 4) << 24); }
// K-major operand (SWIZZLE_32B, layout 6): 16-channel chunk kc of `rows` rows of 32 B, SBO = 256 B per 8-row group
__device__ __forceinline__ uint64_t kdesc(const uint8_t* base, int kc, int rows) { return mdesc(s32(base) + (uint32_t)(kc * rows * 32), 16u, 256u, 6u); }
// MN-major operand (SWIZZLE_128B, layout 2): 64-channel box nb of `rows` rows of 128 B, K-step kc = 16 rows
__device__ __forceinline__ uint64_t ndesc(const uint8_t* base, int nb, int kc, int rows) {
    return mdesc(s32(base) + (uint32_t)(nb * rows * 128 + kc * 16 * 128), (uint32_t)(rows * 128), 1024u, 2u);
}
template <typename T> __device__ __forceinline__ void store_chunk_sw32(uint32_t row_addr, uint32_t sw, const float* e) {
    uint4 lo, hi;
    typename Fmt16<T>::T2* pl = reinterpret_cast<typename Fmt16<T>::T2*>(&lo);
    typename Fmt16<T>::T2* ph = reinterpret_cast<typename Fmt16<T>::T2*>(&hi);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        pl[i] = Fmt16<T>::from_f2(e[2 * i], e[2 * i + 1]);
        ph[i] = Fmt16<T>::from_f2(e[8 + 2 * i], e[8 + 2 * i + 1]);
    }
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(row_addr + (0u ^ sw)), "r"(lo.x), "r"(lo.y), "r"(lo.z), "r"(lo.w) : "memory");
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(row_addr + (16u ^ sw)), "r"(hi.x), "r"(hi.y), "r"(hi.z), "r"(hi.w) : "memory");
}
template <typename T> __device__ __forceinline__ void store_row16(T* dst, const uint32_t* r, float mul) {
    uint4 lo, hi;
    typename Fmt16<T>::T2* pl = reinterpret_cast<typename Fmt16<T>::T2*>(&lo);
    typename Fmt16<T>::T2* ph = reinterpret_cast<typename Fmt16<T>::T2*>(&hi);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        pl[i] = Fmt16<T>::from_f2(__uint_as_float(r[2 * i]) * mul, __uint_as_float(r[2 * i + 1]) * mul);
        ph[i] = Fmt16<T>::from_f2(__uint_as_float(r[8 + 2 * i]) * mul, __uint_as_float(r[8 + 2 * i + 1]) * mul);
    }
    *reinterpret_cast<uint4*>(dst) = lo;
    *reinterpret_cast<uint4*>(dst + 8) = hi;
}
// TMA never writes the rows of a ragged tile past its last token, and the MMAs that reduce over that tile read them as
// the K dimension: stale shared memory there (possibly NaN, and 0 * NaN = NaN) must be zero before the first load.
__device__ __forceinline__ void zero_smem(uint8_t* p, int bytes) {
    for (int i = threadIdx.x * 16; i < bytes; i += ATC_THREADS * 16)
        asm volatile("st.shared.v4.b32 [%0], {%1,%1,%1,%1};" ::"r"(s32(p + i)), "r"(0) : "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// Tiling shared by the three kernels.  The CTA's own tile ("outer": queries of the forward / dq kernel, keys of the dk/dv
// kernel) is R image rows, T = R*W <= 128 tokens, an M = 128 MMA operand.  The loop runs over "inner" tiles of KR rows,
// NK = KR*W tokens, padded to NKp (a multiple of 16) as the MMA's N or K extent.  Tokens are row-major, so tile j
// covers tokens j*NK .. j*NK + NK - 1; the last tile may end past N, and TMA zero-fills its rows past the image.
struct AtGeo {
    int N, W, d, R, T, KR, NK, NKp, nit;
};

struct AtcP {
    TV out; float* lse;
    int heads, inner;
    AtGeo g;
    int nst;                         // K / V stages
    float scale, scale_log2e;
    int q_off, k_off, v_off, p_off, bar_off, kst, vst;   // byte offsets of the shared-memory regions, K / V stage strides
    int zero_v;                      // ragged key tile: zero the V stages once
};

template <typename T, int D>
__global__ void __launch_bounds__(ATC_THREADS, 1) attn_fwd_tc_kernel(const __grid_constant__ CUtensorMap tmQ,
                                                                      const __grid_constant__ CUtensorMap tmK,
                                                                      const __grid_constant__ CUtensorMap tmV, AtcP p) {
    constexpr int KCH = D / 16, NVB = (D + 63) / 64;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* Qs = smem + p.q_off;        // [KCH][128 rows][32 B]     SWIZZLE_32B, K-major
    uint8_t* Ks = smem + p.k_off;        // stages of [KCH][NKp rows][32 B]
    uint8_t* Vs = smem + p.v_off;        // stages of [NVB][NKp rows][128 B]   SWIZZLE_128B, MN-major (64 channels per box)
    uint8_t* Ps = smem + p.p_off;        // [NKp/16][128 rows][32 B]  SWIZZLE_32B, K-major (16 keys per chunk)
    uint64_t* bars = (uint64_t*)(smem + p.bar_off);
    uint64_t *full = bars, *empty = bars + 2, *bar_q = bars + 4, *bar_s = bars + 5, *bar_sfree = bars + 7, *bar_p = bars + 9,
             *bar_o = bars + 10;
    uint32_t* tmem_slot = (uint32_t*)(bars + 11);
    const AtGeo& g = p.g;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int qt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;

    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmQ) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmK) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmV) : "memory");
        for (int i = 0; i < 2; ++i) { mb_init(full + i, 1); mb_init(empty + i, 1); mb_init(bar_s + i, 1); mb_init(bar_sfree + i, 128); }
        mb_init(bar_q, 1); mb_init(bar_p, 128); mb_init(bar_o, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (p.zero_v) zero_smem(Vs, p.nst * p.vst);
    if (warp == 1) tm_alloc(tmem_slot, 512u);
    fence_before();
    __syncthreads();
    fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t o_col = 256u;         // S_j in columns (j & 1) * 128 (an all-keys tile of <= 256 keys: 0..255)

    if (warp == 0) {
        if (lane == 0) {
            mb_expect(bar_q, (uint32_t)(KCH * g.T * 32));
            for (int kc = 0; kc < KCH; ++kc) tma4(Qs + (size_t)kc * 4096, &tmQ, bar_q, h * D + kc * 16, 0, qt * g.R, b);
            for (int j = 0; j < g.nit; ++j) {
                const int s = j % p.nst;
                if (j >= p.nst) mb_wait(empty + s, ((j / p.nst) & 1) ^ 1);
                mb_expect(full + s, (uint32_t)(KCH * g.NK * 32 + NVB * g.NK * 128));
                for (int kc = 0; kc < KCH; ++kc)
                    tma4(Ks + (size_t)s * p.kst + (size_t)kc * g.NKp * 32, &tmK, full + s, p.inner + h * D + kc * 16, 0, j * g.KR, b);
                for (int nb = 0; nb < NVB; ++nb)
                    tma4(Vs + (size_t)s * p.vst + (size_t)nb * g.NKp * 128, &tmV, full + s, 2 * p.inner + h * D + nb * 64, 0, j * g.KR, b);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc1 = idesc_kk<T>(g.NKp), idesc2 = idesc_mn64<T>();
            mb_wait(bar_q, 0);
            // iteration j issues S_j, then P_{j-1} V_{j-1}: the tensor core computes the next scores while the softmax
            // warps exponentiate the current ones
            for (int j = 0; j <= g.nit; ++j) {
                if (j < g.nit) {
                    const int s = j % p.nst;
                    mb_wait(full + s, (j / p.nst) & 1);
                    if (j >= 2) mb_wait(bar_sfree + (j & 1), ((j >> 1) & 1) ^ 1);
                    fence_after();
                    const uint8_t* kb = Ks + (size_t)s * p.kst;
                    for (int kc = 0; kc < KCH; ++kc)
                        mma_f16(tmem_base + (uint32_t)(j & 1) * 128u, kdesc(Qs, kc, 128), kdesc(kb, kc, g.NKp), idesc1, kc > 0 ? 1u : 0u);
                    mma_commit(bar_s + (j & 1));
                }
                if (j >= 1) {
                    const int jp = j - 1, s = jp % p.nst;
                    mb_wait(bar_p, jp & 1);
                    fence_after();
                    const uint8_t* vb = Vs + (size_t)s * p.vst;
                    for (int nb = 0; nb < NVB; ++nb)
                        for (int kc = 0; kc < g.NKp / 16; ++kc)
                            mma_f16(tmem_base + o_col + (uint32_t)nb * 64u, kdesc(Ps, kc, 128), ndesc(vb, nb, kc, g.NKp), idesc2, kc > 0 ? 1u : 0u);
                    mma_commit(bar_o);
                    mma_commit(empty + s);
                }
            }
        }
    } else {
        const int qd = warp & 3;                           // TMEM lane quarter this warp may read
        const int row = qd * 32 + lane;
        const int q = qt * g.T + row;
        const bool valid = row < g.T && q < g.N;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(qd * 32) << 16);
        const uint32_t prow = s32(Ps) + (uint32_t)row * 32u;
        const uint32_t sw = (uint32_t)((row >> 2) & 1) << 4;     // SWIZZLE_32B: 16-byte half index ^= address bit 7
        float o[D];
#pragma unroll
        for (int c = 0; c < D; ++c) o[c] = 0.f;
        float m = -INFINITY, l = 0.f, corr_pend = 0.f;
        // o = o * corr + (P V of the previous tile), read from TMEM once its MMA is complete
        auto fold = [&](float corr) {
#pragma unroll
            for (int c0 = 0; c0 < D; c0 += 16) {
                uint32_t r[16];
                tm_ld16(lane_addr + o_col + (uint32_t)c0, r);
                tm_ld_wait();
#pragma unroll
                for (int i = 0; i < 16; ++i) o[c0 + i] = fmaf(o[c0 + i], corr, __uint_as_float(r[i]));
            }
        };
        for (int j = 0; j < g.nit; ++j) {
            const uint32_t sa = lane_addr + (uint32_t)(j & 1) * 128u;
            const int kv = min(g.NK, g.N - j * g.NK);     // keys of this tile inside the image; the rest are masked to -inf
            mb_wait(bar_s + (j & 1), (j >> 1) & 1);
            fence_after();
            float tmax = -INFINITY;
            for (int c0 = 0; c0 < g.NKp; c0 += 16) {
                uint32_t r[16];
                tm_ld16(sa + (uint32_t)c0, r);
                tm_ld_wait();
#pragma unroll
                for (int i = 0; i < 16; ++i) tmax = fmaxf(tmax, c0 + i < kv ? __uint_as_float(r[i]) : -INFINITY);
            }
            const float m_new = fmaxf(m, tmax);
            const float corr = exp2f((m - m_new) * p.scale_log2e);     // 0 on the first tile (m = -inf)
            if (j > 0) {                                               // P_{j-1} V_{j-1} done: P buffer and O columns free
                mb_wait(bar_o, (j - 1) & 1);
                fence_after();
                fold(corr_pend);
            }
            corr_pend = corr;
            m = m_new;
            const float mb = m * p.scale_log2e;
            float sum = 0.f;
            for (int c0 = 0; c0 < g.NKp; c0 += 16) {
                uint32_t r[16];
                tm_ld16(sa + (uint32_t)c0, r);
                tm_ld_wait();
                float e[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    e[i] = valid && c0 + i < kv ? exp2f(fmaf(__uint_as_float(r[i]), p.scale_log2e, -mb)) : 0.f;
                    sum += e[i];
                }
                store_chunk_sw32<T>(prow + (uint32_t)(c0 >> 4) * 4096u, sw, e);
            }
            l = fmaf(l, corr, sum);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // generic-proxy writes of P -> visible to the tensor core
            fence_before();
            mb_arrive(bar_p);
            mb_arrive(bar_sfree + (j & 1));
        }
        mb_wait(bar_o, (g.nit - 1) & 1);
        fence_after();
        fold(corr_pend);
        {
            const float inv = valid ? 1.0f / l : 0.f;
            const int qq = valid ? q : 0;
            const int y = qq / g.W, x = qq - y * g.W;
            T* orow = p.out.at<T>(b, y, x, h * D);
            if (valid) {
#pragma unroll
                for (int c0 = 0; c0 < D; c0 += 8) {
                    uint4 v;
                    typename Fmt16<T>::T2* pv = reinterpret_cast<typename Fmt16<T>::T2*>(&v);
#pragma unroll
                    for (int i = 0; i < 4; ++i) pv[i] = Fmt16<T>::from_f2(o[c0 + 2 * i] * inv, o[c0 + 2 * i + 1] * inv);
                    *reinterpret_cast<uint4*>(orow + c0) = v;
                }
                p.lse[((size_t)b * p.heads + h) * g.N + q] = m * p.scale + logf(l);
            }
        }
        fence_before();
    }
    __syncthreads();
    if (warp == 1) { fence_after(); tm_dealloc(tmem_base, 512u); }
}


// ------------------------------------------------------------------------------------------------------------------
// Backward, recomputing P from lse (no N x N scratch): two kernels with "natural" operand orientations only.
//
//   dq kernel, one CTA per (image, head, query tile), a loop over key tiles j:   S = Q K_j^T,  dP = dO V_j^T  (TMEM),
//       threads (one query row each): D = dO . O,  P = exp(S*scale - lse),  dS = P * (dP - D)  -> 16-bit K-major chunks,
//       dQ += dS K_j (B = K read MN-major) in TMEM -> * scale -> dqkv[q-channels];  D is also written out for the second kernel.
//   dkv kernel, one CTA per (image, head, key tile), a loop over query tiles i:   S^T = K Q_i^T,  dP^T = V dO_i^T,
//       threads (one key row each): P^T and dS^T from the tile's lse / D (staged in shared memory) -> two 16-bit K-major
//       chunk buffers, dV += P^T dO_i, dK += dS^T Q_i (B = dO / Q read MN-major, loaded into the buffers of the K-major
//       copies once S^T and dP^T are complete) -> dqkv[v-channels], * scale -> dqkv[k-channels].
// TMEM: S at 0, dP at `col_dp`, the accumulators at `col_acc` (after the all-keys tile of N <= 256, over S).
// ------------------------------------------------------------------------------------------------------------------
struct AtbP {
    TV out, dout, dqkv; const float* lse; float* Dbuf;
    int heads, d, inner, kch, nvb;
    AtGeo g;
    int nst, sst;                    // dq kernel: K / V stages and their stride
    float scale, scale_log2e;
    int o0, o1, o2, o3, o4, o5, o6, bar_off;   // byte offsets of the shared-memory regions (see each kernel)
    uint32_t col_dp, col_acc;
    int zero_off, zero_bytes;
};

// regions: o0 Q [kch][128][32], o1 dO [kch][128][32], o2 stages of {K32 [kch][NKp][32], V32 [kch][NKp][32], K128 [nvb][NKp][128]},
//          o5 dS [NKp/16][128][32]
template <typename T>
__global__ void __launch_bounds__(ATC_THREADS, 1) attn_bwd_dq_tc_kernel(const __grid_constant__ CUtensorMap tmQt, const __grid_constant__ CUtensorMap tmGt,
                                                                         const __grid_constant__ CUtensorMap tmF32, const __grid_constant__ CUtensorMap tmF128,
                                                                         AtbP p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t *Qs = smem + p.o0, *Gs = smem + p.o1, *Stg = smem + p.o2, *Ss = smem + p.o5;
    uint64_t* bars = (uint64_t*)(smem + p.bar_off);
    // full: the K-major K / V of a stage (S, dP); full_mn: its MN-major K (dQ), so S and dP need not wait for it
    uint64_t *full = bars, *full_mn = bars + 2, *empty = bars + 4, *bar_in = bars + 6, *bar_s = bars + 7, *bar_ds = bars + 8,
             *bar_o = bars + 9;
    uint32_t* tmem_slot = (uint32_t*)(bars + 10);
    const AtGeo& g = p.g;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int qt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
    const int kbytes = p.kch * g.NKp * 32;           // one K-major copy of a key tile
    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmQt) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmGt) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmF32) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmF128) : "memory");
        for (int i = 0; i < 2; ++i) { mb_init(full + i, 1); mb_init(full_mn + i, 1); mb_init(empty + i, 1); }
        mb_init(bar_in, 1); mb_init(bar_s, 1); mb_init(bar_ds, 128); mb_init(bar_o, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (p.zero_bytes) zero_smem(smem + p.zero_off, p.zero_bytes);
    if (warp == 1) tm_alloc(tmem_slot, 512u);
    fence_before();
    __syncthreads();
    fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (warp == 0) {
        if (lane == 0) {
            mb_expect(bar_in, (uint32_t)(p.kch * 2 * g.T * 32));
            for (int kc = 0; kc < p.kch; ++kc) {
                tma4(Qs + (size_t)kc * 4096, &tmQt, bar_in, h * p.d + kc * 16, 0, qt * g.R, b);
                tma4(Gs + (size_t)kc * 4096, &tmGt, bar_in, h * p.d + kc * 16, 0, qt * g.R, b);
            }
            for (int j = 0; j < g.nit; ++j) {
                const int s = j % p.nst;
                if (j >= p.nst) mb_wait(empty + s, ((j / p.nst) & 1) ^ 1);
                uint8_t* st = Stg + (size_t)s * p.sst;
                mb_expect(full + s, (uint32_t)(p.kch * 2 * g.NK * 32));
                for (int kc = 0; kc < p.kch; ++kc) {
                    tma4(st + (size_t)kc * g.NKp * 32, &tmF32, full + s, p.inner + h * p.d + kc * 16, 0, j * g.KR, b);
                    tma4(st + kbytes + (size_t)kc * g.NKp * 32, &tmF32, full + s, 2 * p.inner + h * p.d + kc * 16, 0, j * g.KR, b);
                }
                mb_expect(full_mn + s, (uint32_t)(p.nvb * g.NK * 128));
                for (int nb = 0; nb < p.nvb; ++nb)
                    tma4(st + 2 * kbytes + (size_t)nb * g.NKp * 128, &tmF128, full_mn + s, p.inner + h * p.d + nb * 64, 0, j * g.KR, b);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc1 = idesc_kk<T>(g.NKp), idesc2 = idesc_mn64<T>();
            mb_wait(bar_in, 0);
            for (int j = 0; j < g.nit; ++j) {
                const int s = j % p.nst;
                const uint8_t* st = Stg + (size_t)s * p.sst;
                mb_wait(full + s, (j / p.nst) & 1);
                fence_after();
                for (int kc = 0; kc < p.kch; ++kc)
                    mma_f16(tmem_base, kdesc(Qs, kc, 128), kdesc(st, kc, g.NKp), idesc1, kc > 0 ? 1u : 0u);
                for (int kc = 0; kc < p.kch; ++kc)
                    mma_f16(tmem_base + p.col_dp, kdesc(Gs, kc, 128), kdesc(st + kbytes, kc, g.NKp), idesc1, kc > 0 ? 1u : 0u);
                mma_commit(bar_s);
                mb_wait(full_mn + s, (j / p.nst) & 1);
                mb_wait(bar_ds, j & 1);              // dS_j written, S_j / dP_j read: their TMEM columns are free again
                fence_after();
                for (int nb = 0; nb < p.nvb; ++nb)
                    for (int kc = 0; kc < g.NKp / 16; ++kc)
                        mma_f16(tmem_base + p.col_acc + (uint32_t)nb * 64u, kdesc(Ss, kc, 128), ndesc(st + 2 * kbytes, nb, kc, g.NKp), idesc2,
                                 (j > 0 || kc > 0) ? 1u : 0u);
                mma_commit(empty + s);
            }
            mma_commit(bar_o);
        }
    } else {
        const int qd = warp & 3, row = qd * 32 + lane;
        const int q = qt * g.T + row;
        const bool valid = row < g.T && q < g.N;
        const int qq = valid ? q : 0;
        const int y = qq / g.W, x = qq - y * g.W;
        // D = dO . O for this query (16-bit token rows of `dout` / `out`), lse of the forward
        float D = 0.f, L = 0.f;
        if (valid) {
            const T* go = p.dout.at<T>(b, y, x, h * p.d);
            const T* oo = p.out.at<T>(b, y, x, h * p.d);
            for (int c = 0; c < p.d; c += 8) {
                const uint4 a = *reinterpret_cast<const uint4*>(go + c), o = *reinterpret_cast<const uint4*>(oo + c);
                const typename Fmt16<T>::T2* ha = reinterpret_cast<const typename Fmt16<T>::T2*>(&a);
                const typename Fmt16<T>::T2* ho = reinterpret_cast<const typename Fmt16<T>::T2*>(&o);
#pragma unroll
                for (int i = 0; i < 4; ++i) { const float2 fa = Fmt16<T>::to_f2(ha[i]), fo = Fmt16<T>::to_f2(ho[i]); D = fmaf(fa.x, fo.x, fmaf(fa.y, fo.y, D)); }
            }
            L = p.lse[((size_t)b * p.heads + h) * g.N + q];
            p.Dbuf[((size_t)b * p.heads + h) * g.N + q] = D;
        }
        const float Lb = L * 1.4426950408889634f;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(qd * 32) << 16);
        const uint32_t srow = s32(Ss) + (uint32_t)row * 32u, sw = (uint32_t)((row >> 2) & 1) << 4;
        for (int j = 0; j < g.nit; ++j) {
            const int kv = min(g.NK, g.N - j * g.NK);
            mb_wait(bar_s, j & 1);                   // also: dQ += dS_{j-1} K_{j-1} is complete, the dS buffer is free
            fence_after();
            for (int c0 = 0; c0 < g.NKp; c0 += 16) {
                uint32_t rs[16], rp[16];
                tm_ld16(lane_addr + (uint32_t)c0, rs);
                tm_ld16(lane_addr + p.col_dp + (uint32_t)c0, rp);
                tm_ld_wait();
                float e[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const float pij = exp2f(fmaf(__uint_as_float(rs[i]), p.scale_log2e, -Lb));
                    e[i] = valid && c0 + i < kv ? pij * (__uint_as_float(rp[i]) - D) : 0.f;
                }
                store_chunk_sw32<T>(srow + (uint32_t)(c0 >> 4) * 4096u, sw, e);
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            fence_before();
            mb_arrive(bar_ds);
        }
        mb_wait(bar_o, 0);
        fence_after();
        T* drow = p.dqkv.at<T>(b, y, x, h * p.d);
        for (int c0 = 0; c0 < p.d; c0 += 16) {
            uint32_t r[16];
            tm_ld16(lane_addr + p.col_acc + (uint32_t)c0, r);
            tm_ld_wait();
            if (valid) store_row16<T>(drow + c0, r, p.scale);
        }
        fence_before();
    }
    __syncthreads();
    if (warp == 1) { fence_after(); tm_dealloc(tmem_base, 512u); }
}

// regions: o0 K tile [kch][128][32], o1 V tile [kch][128][32], o2 Q32 [kch][NKp][32] then Q128 [nvb][NKp][128],
//          o3 dO32 then dO128 likewise, o4 P^T [NKp/16][128][32], o5 dS^T likewise, o6 the query tile's lse / D [2][NKp]
//          (inside the dead K tile when there is a single query tile)
template <typename T>
__global__ void __launch_bounds__(ATC_THREADS, 1) attn_bwd_dkv_tc_kernel(const __grid_constant__ CUtensorMap tmKt, const __grid_constant__ CUtensorMap tmQ32,
                                                                          const __grid_constant__ CUtensorMap tmG32, const __grid_constant__ CUtensorMap tmQ128,
                                                                          const __grid_constant__ CUtensorMap tmG128, AtbP p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t *Kt = smem + p.o0, *Vt = smem + p.o1, *Qr = smem + p.o2, *Gr = smem + p.o3, *Pt = smem + p.o4, *St = smem + p.o5;
    uint64_t* bars = (uint64_t*)(smem + p.bar_off);
    uint64_t *bar_kv = bars, *bar_in = bars + 1, *bar_in2 = bars + 2, *bar_s = bars + 3, *bar_p = bars + 4, *bar_free = bars + 5,
             *bar_o = bars + 6;
    uint32_t* tmem_slot = (uint32_t*)(bars + 7);
    const AtGeo& g = p.g;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int kt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmKt) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmQ32) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmG32) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmQ128) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmG128) : "memory");
        mb_init(bar_kv, 1); mb_init(bar_in, 1); mb_init(bar_in2, 1); mb_init(bar_s, 1); mb_init(bar_p, 128); mb_init(bar_free, 1);
        mb_init(bar_o, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (p.zero_bytes) zero_smem(smem + p.zero_off, p.zero_bytes);
    if (warp == 1) tm_alloc(tmem_slot, 512u);
    fence_before();
    __syncthreads();
    fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (warp == 0) {
        if (lane == 0) {
            mb_expect(bar_kv, (uint32_t)(p.kch * 2 * g.T * 32));
            for (int kc = 0; kc < p.kch; ++kc) {
                tma4(Kt + (size_t)kc * 4096, &tmKt, bar_kv, p.inner + h * p.d + kc * 16, 0, kt * g.R, b);
                tma4(Vt + (size_t)kc * 4096, &tmKt, bar_kv, 2 * p.inner + h * p.d + kc * 16, 0, kt * g.R, b);
            }
            for (int i = 0; i < g.nit; ++i) {
                if (i > 0) mb_wait(bar_free, (i - 1) & 1);      // dV / dK of the previous query tile no longer read Q, dO
                mb_expect(bar_in, (uint32_t)(p.kch * 2 * g.NK * 32));
                for (int kc = 0; kc < p.kch; ++kc) {
                    tma4(Qr + (size_t)kc * g.NKp * 32, &tmQ32, bar_in, h * p.d + kc * 16, 0, i * g.KR, b);
                    tma4(Gr + (size_t)kc * g.NKp * 32, &tmG32, bar_in, h * p.d + kc * 16, 0, i * g.KR, b);
                }
                // the MN-major copies of Q and dO replace the K-major ones once S^T and dP^T are complete
                mb_wait(bar_s, i & 1);
                mb_expect(bar_in2, (uint32_t)(p.nvb * 2 * g.NK * 128));
                for (int nb = 0; nb < p.nvb; ++nb) {
                    tma4(Qr + (size_t)nb * g.NKp * 128, &tmQ128, bar_in2, h * p.d + nb * 64, 0, i * g.KR, b);
                    tma4(Gr + (size_t)nb * g.NKp * 128, &tmG128, bar_in2, h * p.d + nb * 64, 0, i * g.KR, b);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc1 = idesc_kk<T>(g.NKp), idesc2 = idesc_mn64<T>();
            const uint32_t col_dv = p.col_acc, col_dk = p.col_acc + (uint32_t)p.nvb * 64u;
            mb_wait(bar_kv, 0);
            for (int i = 0; i < g.nit; ++i) {
                mb_wait(bar_in, i & 1);
                fence_after();
                for (int kc = 0; kc < p.kch; ++kc)
                    mma_f16(tmem_base, kdesc(Kt, kc, 128), kdesc(Qr, kc, g.NKp), idesc1, kc > 0 ? 1u : 0u);
                for (int kc = 0; kc < p.kch; ++kc)
                    mma_f16(tmem_base + p.col_dp, kdesc(Vt, kc, 128), kdesc(Gr, kc, g.NKp), idesc1, kc > 0 ? 1u : 0u);
                mma_commit(bar_s);
                mb_wait(bar_in2, i & 1);
                mb_wait(bar_p, i & 1);
                fence_after();
                for (int nb = 0; nb < p.nvb; ++nb)
                    for (int kc = 0; kc < g.NKp / 16; ++kc)        // dV += P^T dO
                        mma_f16(tmem_base + col_dv + (uint32_t)nb * 64u, kdesc(Pt, kc, 128), ndesc(Gr, nb, kc, g.NKp), idesc2,
                                 (i > 0 || kc > 0) ? 1u : 0u);
                for (int nb = 0; nb < p.nvb; ++nb)
                    for (int kc = 0; kc < g.NKp / 16; ++kc)        // dK += dS^T Q
                        mma_f16(tmem_base + col_dk + (uint32_t)nb * 64u, kdesc(St, kc, 128), ndesc(Qr, nb, kc, g.NKp), idesc2,
                                 (i > 0 || kc > 0) ? 1u : 0u);
                mma_commit(bar_free);
            }
            mma_commit(bar_o);
        }
    } else {
        const int qd = warp & 3, row = qd * 32 + lane;
        const int j = kt * g.T + row;
        const bool valid = row < g.T && j < g.N;
        const int jj = valid ? j : 0;
        const int y = jj / g.W, x = jj - y * g.W;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(qd * 32) << 16);
        const uint32_t prow = s32(Pt) + (uint32_t)row * 32u, srow = s32(St) + (uint32_t)row * 32u, sw = (uint32_t)((row >> 2) & 1) << 4;
        float* Ls = reinterpret_cast<float*>(smem + p.o6);
        float* Ds = Ls + g.NKp;
        const size_t bh = ((size_t)b * p.heads + h) * g.N;
        for (int i = 0; i < g.nit; ++i) {
            const int nq = min(g.NK, g.N - i * g.NK);
            mb_wait(bar_s, i & 1);                         // S^T, dP^T complete (and with them the previous dV / dK MMAs)
            fence_after();
            asm volatile("bar.sync 1, 128;" ::: "memory");  // every thread is done with the previous tile's lse / D
            for (int c = threadIdx.x - 64; c < g.NKp; c += 128) {
                const bool ok = c < nq;
                Ls[c] = ok ? p.lse[bh + i * g.NK + c] * 1.4426950408889634f : 0.f;
                Ds[c] = ok ? p.Dbuf[bh + i * g.NK + c] : 0.f;
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");
            for (int c0 = 0; c0 < g.NKp; c0 += 16) {
                uint32_t rs[16], rp[16];
                tm_ld16(lane_addr + (uint32_t)c0, rs);
                tm_ld16(lane_addr + p.col_dp + (uint32_t)c0, rp);
                tm_ld_wait();
                float e[16], f[16];
#pragma unroll
                for (int k = 0; k < 16; ++k) {
                    const bool ok = valid && c0 + k < nq;
                    const float pij = ok ? exp2f(fmaf(__uint_as_float(rs[k]), p.scale_log2e, -Ls[c0 + k])) : 0.f;
                    e[k] = pij;
                    f[k] = ok ? pij * (__uint_as_float(rp[k]) - Ds[c0 + k]) : 0.f;
                }
                store_chunk_sw32<T>(prow + (uint32_t)(c0 >> 4) * 4096u, sw, e);
                store_chunk_sw32<T>(srow + (uint32_t)(c0 >> 4) * 4096u, sw, f);
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            fence_before();
            mb_arrive(bar_p);
        }
        mb_wait(bar_o, 0);
        fence_after();
        T* krow = p.dqkv.at<T>(b, y, x, p.inner + h * p.d);
        T* vrow = p.dqkv.at<T>(b, y, x, 2 * p.inner + h * p.d);
        for (int c0 = 0; c0 < p.d; c0 += 16) {
            uint32_t rv[16], rk[16];
            tm_ld16(lane_addr + p.col_acc + (uint32_t)c0, rv);
            tm_ld16(lane_addr + p.col_acc + (uint32_t)p.nvb * 64u + (uint32_t)c0, rk);
            tm_ld_wait();
            if (valid) { store_row16<T>(vrow + c0, rv, 1.0f); store_row16<T>(krow + c0, rk, p.scale); }
        }
        fence_before();
    }
    __syncthreads();
    if (warp == 1) { fence_after(); tm_dealloc(tmem_base, 512u); }
}

}  // namespace

#define ATC_SMEM_MAX (227 * 1024)

static AtGeo atc_geo(const ddpm_tensor* t, int d) {
    AtGeo g;
    g.N = t->H * t->W; g.W = t->W; g.d = d;
    g.R = 128 / t->W < t->H ? 128 / t->W : t->H;
    g.T = g.R * t->W;
    // one all-keys tile for N <= 256 at head_dim <= 64 (S and dP of 256 keys fill the TMEM, its shared memory fits)
    g.KR = g.N <= 256 && d <= 64 ? t->H : g.R;
    g.NK = g.KR * t->W;
    g.NKp = (g.NK + 15) & ~15;
    g.nit = (t->H + g.KR - 1) / g.KR;
    return g;
}

static int atc_smem_attr(const void* kernel, size_t smem) {
    if (smem > ATC_SMEM_MAX) return DDPM_E_ARG;
    return (int)cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
}

// bf16 / fp16; head_dim 32 / 64 / 128 (V, dO, Q are read as 64-channel boxes: with head_dim 32 the upper 32 output columns are
// the next head's and are ignored); W <= 128 so that a tile holds at least one whole image row.
int attn_tc_supported(const ddpm_tensor* qkv, const ddpm_tensor* out, int heads, int d, int dtype) {
    if ((dtype != DDPM_BF16 && dtype != DDPM_F16) || (d != 32 && d != 64 && d != 128)) return 0;
    if (qkv->W > 128) return 0;
    if (qkv->halo != 1 && qkv->halo != 0) return 0;
    if (qkv->pitch % 8 || out->pitch % 8 || ((uintptr_t)qkv->ptr & 15) || ((uintptr_t)out->ptr & 15)) return 0;
    if ((heads * d) % 8) return 0;
    return 1;
}

// 4-D tensor map over (channel, x, y, image) of one NHWC 16-bit tensor, halo excluded: boxes of `channels` x W x `rows`,
// 16 channels SWIZZLE_32B (K-major operands), 64 channels SWIZZLE_128B (MN-major operands)
template <typename T>
static int atc_map(const ddpm_tensor* t, int channels, int rows, CUtensorMap* m) {
    const int Hp = t->H + 2 * t->halo, Wp = t->W + 2 * t->halo;
    char* base = (char*)t->ptr + ((size_t)t->halo * Wp + t->halo) * t->pitch * 2;
    const uint64_t dims[4] = {(uint64_t)t->C, (uint64_t)t->W, (uint64_t)t->H, (uint64_t)t->N};
    const uint64_t strides[3] = {(uint64_t)t->pitch * 2, (uint64_t)Wp * t->pitch * 2, (uint64_t)Hp * Wp * t->pitch * 2};
    const uint32_t box[4] = {(uint32_t)channels, (uint32_t)t->W, (uint32_t)rows, 1u};
    return ddpm_encode_tiled16(m, Fmt16<T>::tma_type, base, 4, dims, strides, box, channels == 16 ? 32 : 128);
}

template <typename T, int D>
static int attn_fwd_tc_launch(const ddpm_tensor* qkv, AtcP& p, cudaStream_t st) {
    const AtGeo& g = p.g;
    constexpr int KCH = D / 16, NVB = (D + 63) / 64;
    p.nst = g.nit > 1 ? 2 : 1;
    p.kst = KCH * g.NKp * 32;
    p.vst = NVB * g.NKp * 128;
    p.q_off = 0;
    p.k_off = KCH * 4096;
    p.v_off = (p.k_off + p.nst * p.kst + 1023) & ~1023;
    p.p_off = (p.v_off + p.nst * p.vst + 1023) & ~1023;
    p.bar_off = p.p_off + (g.NKp / 16) * 4096;
    p.zero_v = g.NK != g.NKp;
    const size_t smem = (size_t)p.bar_off + 8 * 11 + 16 + 1024;
    CUtensorMap tmQ, tmK, tmV;
    int rc = atc_map<T>(qkv, 16, g.R, &tmQ); if (rc) return rc;
    rc = atc_map<T>(qkv, 16, g.KR, &tmK); if (rc) return rc;
    rc = atc_map<T>(qkv, 64, g.KR, &tmV); if (rc) return rc;
    static size_t configured = 0;
    if (smem > configured) { rc = atc_smem_attr((const void*)attn_fwd_tc_kernel<T, D>, smem); if (rc) return rc; configured = smem; }
    dim3 grid((qkv->H + g.R - 1) / g.R, p.heads, qkv->N);
    CUDA_TRY(launch_kernel(attn_fwd_tc_kernel<T, D>, grid, dim3(ATC_THREADS), smem, st, tmQ, tmK, tmV, p));
    LAUNCH_OK();
    return 0;
}

template <typename T>
static int attn_tc_launch_t(const ddpm_tensor* qkv, const ddpm_tensor* out, int heads, int d, float* lse, cudaStream_t st) {
    AtcP p;
    p.out = TV(*out); p.lse = lse; p.heads = heads; p.inner = heads * d;
    p.g = atc_geo(qkv, d);
    p.scale = 1.0f / sqrtf((float)d); p.scale_log2e = p.scale * 1.4426950408889634f;
    if (d == 32) return attn_fwd_tc_launch<T, 32>(qkv, p, st);
    if (d == 64) return attn_fwd_tc_launch<T, 64>(qkv, p, st);
    return attn_fwd_tc_launch<T, 128>(qkv, p, st);
}

int attn_tc_launch(const ddpm_tensor* qkv, const ddpm_tensor* out, int heads, int d, float* lse, int dtype, cudaStream_t st) {
    if (dtype == DDPM_BF16) return attn_tc_launch_t<bf16>(qkv, out, heads, d, lse, st);
    if (dtype == DDPM_F16) return attn_tc_launch_t<f16>(qkv, out, heads, d, lse, st);
    return DDPM_E_ARG;
}

// floats of scratch the tensor-core backward needs (D = dO . O per query) -- 0 when the shape is not eligible
int64_t attn_tc_bwd_scratch_floats(const ddpm_tensor* qkv, const ddpm_tensor* out, int heads, int d, int dtype) {
    if (!attn_tc_supported(qkv, out, heads, d, dtype)) return 0;
    return (int64_t)qkv->N * heads * qkv->H * qkv->W;
}

template <typename T>
static int attn_tc_bwd_launch_t(const ddpm_tensor* qkv, const ddpm_tensor* out, const ddpm_tensor* dout, const float* lse,
                                const ddpm_tensor* dqkv, int heads, int d, float* scratch, cudaStream_t st) {
    AtbP p;
    p.out = TV(*out); p.dout = TV(*dout); p.dqkv = TV(*dqkv); p.lse = lse; p.Dbuf = scratch;
    p.heads = heads; p.d = d; p.inner = heads * d; p.kch = d / 16; p.nvb = (d + 63) / 64;
    p.g = atc_geo(qkv, d);
    const AtGeo& g = p.g;
    p.scale = 1.0f / sqrtf((float)d); p.scale_log2e = p.scale * 1.4426950408889634f;
    // S at 0 and dP after it; with several inner tiles the accumulators take columns 256.., with one they reuse S's
    p.col_dp = g.NKp > 128 ? 256u : 128u;
    p.col_acc = g.nit > 1 ? 256u : 0u;
    const bool ragged = g.NK != g.NKp;
    const int A1 = p.kch * 4096, K32 = p.kch * g.NKp * 32, M128 = p.nvb * g.NKp * 128, CH = (g.NKp / 16) * 4096;
    CUtensorMap qT, qF32, qF128, gT, gF32, gF128;
    int rc = atc_map<T>(qkv, 16, g.R, &qT); if (rc) return rc;
    if ((rc = atc_map<T>(qkv, 16, g.KR, &qF32)) || (rc = atc_map<T>(qkv, 64, g.KR, &qF128))) return rc;
    if ((rc = atc_map<T>(dout, 16, g.R, &gT)) || (rc = atc_map<T>(dout, 16, g.KR, &gF32)) || (rc = atc_map<T>(dout, 64, g.KR, &gF128))) return rc;
    dim3 grid((qkv->H + g.R - 1) / g.R, heads, qkv->N);
    {   // dq: Q, dO, stages of {K32, V32, K128}, dS
        p.sst = (2 * K32 + M128 + 1023) & ~1023;
        p.o0 = 0; p.o1 = A1; p.o2 = 2 * A1;
        p.nst = g.nit > 1 && (size_t)p.o2 + 2 * p.sst + CH + 8 * 10 + 16 + 1024 <= ATC_SMEM_MAX ? 2 : 1;
        p.o5 = p.o2 + p.nst * p.sst;
        p.bar_off = p.o5 + CH;
        p.zero_off = p.o2; p.zero_bytes = ragged ? p.nst * p.sst : 0;
        const size_t smem = (size_t)p.bar_off + 8 * 10 + 16 + 1024;
        static size_t configured = 0;
        if (smem > configured) { rc = atc_smem_attr((const void*)attn_bwd_dq_tc_kernel<T>, smem); if (rc) return rc; configured = smem; }
        CUDA_TRY(launch_kernel(attn_bwd_dq_tc_kernel<T>, grid, dim3(ATC_THREADS), smem, st, qT, gT, qF32, qF128, p));
        LAUNCH_OK();
    }
    {   // dkv: K tile, V tile, Q32 -> Q128, dO32 -> dO128, P^T, dS^T, lse / D of the query tile
        const int RB = (K32 > M128 ? K32 : M128);
        p.o0 = 0; p.o1 = A1; p.o2 = 2 * A1; p.o3 = p.o2 + RB; p.o4 = p.o3 + RB; p.o5 = p.o4 + CH;
        p.o6 = g.nit == 1 ? 0 : p.o5 + CH;
        p.bar_off = (g.nit == 1 ? p.o5 + CH : p.o6 + 2 * g.NKp * 4 + 7) & ~7;
        p.zero_off = p.o2; p.zero_bytes = ragged ? 2 * RB : 0;
        const size_t smem = (size_t)p.bar_off + 8 * 7 + 16 + 1024;
        static size_t configured = 0;
        if (smem > configured) { rc = atc_smem_attr((const void*)attn_bwd_dkv_tc_kernel<T>, smem); if (rc) return rc; configured = smem; }
        CUDA_TRY(launch_kernel(attn_bwd_dkv_tc_kernel<T>, grid, dim3(ATC_THREADS), smem, st, qT, qF32, gF32, qF128, gF128, p));
        LAUNCH_OK();
    }
    return 0;
}

int attn_tc_bwd_launch(const ddpm_tensor* qkv, const ddpm_tensor* out, const ddpm_tensor* dout, const float* lse,
                       const ddpm_tensor* dqkv, int heads, int d, float* scratch, int dtype, cudaStream_t st) {
    if (dtype == DDPM_BF16) return attn_tc_bwd_launch_t<bf16>(qkv, out, dout, lse, dqkv, heads, d, scratch, st);
    if (dtype == DDPM_F16) return attn_tc_bwd_launch_t<f16>(qkv, out, dout, lse, dqkv, heads, d, scratch, st);
    return DDPM_E_ARG;
}
