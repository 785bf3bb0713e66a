// tcgen05 / TMEM forward of the spatial self-attention block (attention.py:56-74) for the shapes the UNets use:
// N = H*W <= 256 tokens, head_dim 32 or 64, bf16.  One CTA per (image, head, 128-query tile):
//
//   S = Q K^T      tcgen05.mma, M = 128 queries, N = all keys (<= 256), K = head_dim; Q and K arrive by TMA straight out of
//                  the NHWC `qkv` tensor (4-D maps over (channel, x, y, image): the halo pixels are not in the box, the
//                  permute + contiguous copies of attention.py:63-65 never exist) as 16-channel K-major chunks, SWIZZLE_32B;
//                  S lives in tensor memory (<= 256 fp32 columns)
//   P = softmax    128 threads, one query row each: two passes over their TMEM lane (max, then exp2 + sum), P written as
//                  bf16 into shared memory in the same 16-key K-major chunk layout (single pass: N <= 256 needs no online
//                  rescaling)
//   O = P V        second tcgen05.mma, A = P (K-major), B = V read MN-major (head_dim contiguous, SWIZZLE_128B) exactly as it
//                  sits in `qkv`; O in TMEM columns 256.., scaled by 1/rowsum in the epilogue and stored as bf16 token rows
//                  (the permute back, attention.py:72, is the store address); lse = max*scale + log(sum) for the backward.
//
// Attention is <0.4 % of the model FLOPs but 6 % of the CelebA256 step with the CUDA-core kernels of attn_kernels.cu
// (profiles/r2_launches_step_celeba256_summary.txt); those remain the fp32 path, the backward and the fallback for other
// shapes.
#include "common.cuh"
#include <cuda.h>
#include <cudaTypedefs.h>
#include <math.h>

extern int ddpm_encode_tiled_bf16(CUtensorMap* m, void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                                  const uint32_t* box, int swizzle_bytes);      // conv_tc.cu

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
__device__ __forceinline__ void mma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
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

struct AtcP {
    TV out; float* lse;
    int heads, d, inner, N, NK;      // tokens per image (queries) and keys (= N)
    int tok_q, rows_q;               // queries per CTA tile (<= 128) and the image rows they span
    int kch;                         // 16-channel chunks of the head dimension
    int W;
    float scale, scale_log2e;
    int q_off, k_off, v_off, p_off;  // byte offsets of the operand tiles in shared memory
};

__global__ void __launch_bounds__(ATC_THREADS, 1) attn_fwd_tc_kernel(const __grid_constant__ CUtensorMap tmQ,
                                                                      const __grid_constant__ CUtensorMap tmK,
                                                                      const __grid_constant__ CUtensorMap tmV, AtcP p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* Qs = smem + p.q_off;        // [kch][128 rows][32 B]   SWIZZLE_32B, K-major
    uint8_t* Ks = smem + p.k_off;        // [kch][NK rows][32 B]
    uint8_t* Vs = smem + p.v_off;        // [NK rows][128 B]        SWIZZLE_128B, MN-major (64 channels)
    uint8_t* Ps = smem + p.p_off;        // [NK/16][128 rows][32 B] SWIZZLE_32B, K-major (16 keys per chunk)
    uint64_t* bars = (uint64_t*)(Ps + (size_t)(p.NK / 16) * 4096);
    uint64_t* bar_qk = bars; uint64_t* bar_v = bars + 1; uint64_t* bar_s = bars + 2; uint64_t* bar_p = bars + 3; uint64_t* bar_o = bars + 4;
    uint32_t* tmem_slot = (uint32_t*)(bars + 5);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int qt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;

    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmQ) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmK) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmV) : "memory");
        mb_init(bar_qk, 1); mb_init(bar_v, 1); mb_init(bar_s, 1); mb_init(bar_p, 128); mb_init(bar_o, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tm_alloc(tmem_slot, 512u);
    fence_before();
    __syncthreads();
    fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t o_col = 256u;

    if (warp == 0) {
        if (lane == 0) {
            mb_expect(bar_qk, (uint32_t)(p.kch * (p.tok_q + p.NK) * 32));
            for (int kc = 0; kc < p.kch; ++kc) {
                tma4(Qs + (size_t)kc * 4096, &tmQ, bar_qk, h * p.d + kc * 16, 0, qt * p.rows_q, b);
                tma4(Ks + (size_t)kc * p.NK * 32, &tmK, bar_qk, p.inner + h * p.d + kc * 16, 0, 0, b);
            }
            mb_expect(bar_v, (uint32_t)(p.NK * 128));
            tma4(Vs, &tmV, bar_v, 2 * p.inner + h * p.d, 0, 0, b);
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // S = Q K^T: K-major operands, SWIZZLE_32B (layout 6), SBO = 256 B per 8-row group -- the recipe of conv_tc2's A/B tiles
            const uint32_t idesc1 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.NK >> 3) << 17) | ((128u >> 4) << 24);
            mb_wait(bar_qk, 0);
            fence_after();
            for (int kc = 0; kc < p.kch; ++kc)
                mma_bf16(tmem_base, mdesc(s32(Qs) + (uint32_t)kc * 4096u, 16u, 256u, 6u),
                         mdesc(s32(Ks) + (uint32_t)(kc * p.NK * 32), 16u, 256u, 6u), idesc1, kc > 0 ? 1u : 0u);
            mma_commit(bar_s);
            // O = P V: A = P (K-major, SWIZZLE_32B), B = V MN-major (bit 16), SWIZZLE_128B (layout 2), SBO = 1024 B -- wgrad's recipe
            const uint32_t idesc2 = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((64u >> 3) << 17) | ((128u >> 4) << 24);
            mb_wait(bar_v, 0);
            mb_wait(bar_p, 0);
            fence_after();
            for (int kc = 0; kc < p.NK / 16; ++kc)
                mma_bf16(tmem_base + o_col, mdesc(s32(Ps) + (uint32_t)kc * 4096u, 16u, 256u, 6u),
                         mdesc(s32(Vs) + (uint32_t)(kc * 16 * 128), (uint32_t)(p.NK * 128), 1024u, 2u), idesc2, kc > 0 ? 1u : 0u);
            mma_commit(bar_o);
        }
    } else {
        const int qd = warp & 3;                           // TMEM lane quarter this warp may read
        const int row = qd * 32 + lane;
        const int q = qt * p.tok_q + row;
        const bool valid = row < p.tok_q && q < p.N;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(qd * 32) << 16);
        mb_wait(bar_s, 0);
        fence_after();
        float m = -INFINITY;
        for (int c0 = 0; c0 < p.NK; c0 += 16) {
            uint32_t r[16];
            tm_ld16(lane_addr + (uint32_t)c0, r);
            tm_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) m = fmaxf(m, __uint_as_float(r[i]));
        }
        if (!valid) m = 0.f;
        const float mb = m * p.scale_log2e;
        float sum = 0.f;
        const uint32_t prow = s32(Ps) + (uint32_t)row * 32u;
        const uint32_t sw = (uint32_t)((row >> 2) & 1) << 4;     // SWIZZLE_32B: 16-byte half index ^= address bit 7
        for (int c0 = 0; c0 < p.NK; c0 += 16) {
            uint32_t r[16];
            tm_ld16(lane_addr + (uint32_t)c0, r);
            tm_ld_wait();
            float e[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                e[i] = valid ? exp2f(fmaf(__uint_as_float(r[i]), p.scale_log2e, -mb)) : 0.f;
                sum += e[i];
            }
            uint4 lo, hi;
            __nv_bfloat162* pl = reinterpret_cast<__nv_bfloat162*>(&lo);
            __nv_bfloat162* ph = reinterpret_cast<__nv_bfloat162*>(&hi);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                pl[i] = __floats2bfloat162_rn(e[2 * i], e[2 * i + 1]);
                ph[i] = __floats2bfloat162_rn(e[8 + 2 * i], e[8 + 2 * i + 1]);
            }
            const uint32_t base = prow + (uint32_t)(c0 >> 4) * 4096u;
            asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(base + (0u ^ sw)), "r"(lo.x), "r"(lo.y), "r"(lo.z), "r"(lo.w) : "memory");
            asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(base + (16u ^ sw)), "r"(hi.x), "r"(hi.y), "r"(hi.z), "r"(hi.w) : "memory");
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // generic-proxy writes of P -> visible to the tensor core
        fence_before();
        mb_arrive(bar_p);
        mb_wait(bar_o, 0);
        fence_after();
        {
            const float inv = valid ? 1.0f / sum : 0.f;
            const int qq = valid ? q : 0;
            const int y = qq / p.W, x = qq - y * p.W;
            bf16* orow = p.out.at<bf16>(b, y, x, h * p.d);
            for (int c0 = 0; c0 < p.d; c0 += 16) {
                uint32_t r[16];
                tm_ld16(lane_addr + o_col + (uint32_t)c0, r);       // warp-collective: every lane loads, valid rows store
                tm_ld_wait();
                uint4 lo, hi;
                __nv_bfloat162* pl = reinterpret_cast<__nv_bfloat162*>(&lo);
                __nv_bfloat162* ph = reinterpret_cast<__nv_bfloat162*>(&hi);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    pl[i] = __floats2bfloat162_rn(__uint_as_float(r[2 * i]) * inv, __uint_as_float(r[2 * i + 1]) * inv);
                    ph[i] = __floats2bfloat162_rn(__uint_as_float(r[8 + 2 * i]) * inv, __uint_as_float(r[8 + 2 * i + 1]) * inv);
                }
                if (valid) {
                    *reinterpret_cast<uint4*>(orow + c0) = lo;
                    *reinterpret_cast<uint4*>(orow + c0 + 8) = hi;
                }
            }
            if (valid) p.lse[((size_t)b * p.heads + h) * p.N + q] = m * p.scale + logf(sum);
        }
        fence_before();
    }
    __syncthreads();
    if (warp == 1) { fence_after(); tm_dealloc(tmem_base, 512u); }
}


// ------------------------------------------------------------------------------------------------------------------
// Backward, recomputing P from lse (no N x N scratch): two kernels with "natural" operand orientations only.
//
//   dq kernel, one CTA per (image, head, 128-query tile):   S = Q K^T,  dP = dO V^T  (both into TMEM, 2 x <=256 columns),
//       threads (one query row each): D = dO . O,  P = exp(S*scale - lse),  dS = P * (dP - D)  -> bf16 K-major chunks,
//       dQ = dS K (B = K read MN-major) -> * scale -> dqkv[q-channels];  D is also written out for the second kernel.
//   dkv kernel, one CTA per (image, head, 128-key tile):     S^T = K Q^T,  dP^T = V dO^T,
//       threads (one key row each): P^T and dS^T from the per-query lse / D  -> two bf16 K-major chunk buffers,
//       dV = P^T dO,  dK = dS^T Q (B = dO / Q read MN-major) -> dqkv[v-channels], * scale -> dqkv[k-channels].
// ------------------------------------------------------------------------------------------------------------------
struct AtbP {
    TV out, dout, dqkv; const float* lse; float* Dbuf;
    int heads, d, inner, N, tok_t, rows_t, kch, W;
    float scale, scale_log2e;
    int o0, o1, o2, o3, o4, o5;      // byte offsets of the shared-memory regions (see each kernel)
};
__device__ __forceinline__ void store_chunk_sw32(uint32_t row_addr, uint32_t sw, const float* e) {
    uint4 lo, hi;
    __nv_bfloat162* pl = reinterpret_cast<__nv_bfloat162*>(&lo);
    __nv_bfloat162* ph = reinterpret_cast<__nv_bfloat162*>(&hi);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        pl[i] = __floats2bfloat162_rn(e[2 * i], e[2 * i + 1]);
        ph[i] = __floats2bfloat162_rn(e[8 + 2 * i], e[8 + 2 * i + 1]);
    }
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(row_addr + (0u ^ sw)), "r"(lo.x), "r"(lo.y), "r"(lo.z), "r"(lo.w) : "memory");
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(row_addr + (16u ^ sw)), "r"(hi.x), "r"(hi.y), "r"(hi.z), "r"(hi.w) : "memory");
}
__device__ __forceinline__ void store_row16(bf16* dst, const uint32_t* r, float mul) {
    uint4 lo, hi;
    __nv_bfloat162* pl = reinterpret_cast<__nv_bfloat162*>(&lo);
    __nv_bfloat162* ph = reinterpret_cast<__nv_bfloat162*>(&hi);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        pl[i] = __floats2bfloat162_rn(__uint_as_float(r[2 * i]) * mul, __uint_as_float(r[2 * i + 1]) * mul);
        ph[i] = __floats2bfloat162_rn(__uint_as_float(r[8 + 2 * i]) * mul, __uint_as_float(r[8 + 2 * i + 1]) * mul);
    }
    *reinterpret_cast<uint4*>(dst) = lo;
    *reinterpret_cast<uint4*>(dst + 8) = hi;
}

// regions: o0 Q [kch][128][32], o1 dO [kch][128][32], o2 K32 [kch][N][32], o3 V32 [kch][N][32], o4 K128 [N][128], o5 dS [N/16][128][32]
__global__ void __launch_bounds__(ATC_THREADS, 1) attn_bwd_dq_tc_kernel(const __grid_constant__ CUtensorMap tmQt, const __grid_constant__ CUtensorMap tmGt,
                                                                         const __grid_constant__ CUtensorMap tmF32, const __grid_constant__ CUtensorMap tmF128,
                                                                         AtbP p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t *Qs = smem + p.o0, *Gs = smem + p.o1, *K32 = smem + p.o2, *V32 = smem + p.o3, *K128 = smem + p.o4, *Ss = smem + p.o5;
    uint64_t* bars = (uint64_t*)(Ss + (size_t)(p.N / 16) * 4096);
    uint64_t *bar_in = bars, *bar_k = bars + 1, *bar_s = bars + 2, *bar_ds = bars + 3, *bar_o = bars + 4;
    uint32_t* tmem_slot = (uint32_t*)(bars + 5);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int qt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmQt) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmGt) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmF32) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmF128) : "memory");
        mb_init(bar_in, 1); mb_init(bar_k, 1); mb_init(bar_s, 1); mb_init(bar_ds, 128); mb_init(bar_o, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tm_alloc(tmem_slot, 512u);
    fence_before();
    __syncthreads();
    fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (warp == 0) {
        if (lane == 0) {
            mb_expect(bar_in, (uint32_t)(p.kch * (2 * p.tok_t + 2 * p.N) * 32));
            for (int kc = 0; kc < p.kch; ++kc) {
                tma4(Qs + (size_t)kc * 4096, &tmQt, bar_in, h * p.d + kc * 16, 0, qt * p.rows_t, b);
                tma4(Gs + (size_t)kc * 4096, &tmGt, bar_in, h * p.d + kc * 16, 0, qt * p.rows_t, b);
                tma4(K32 + (size_t)kc * p.N * 32, &tmF32, bar_in, p.inner + h * p.d + kc * 16, 0, 0, b);
                tma4(V32 + (size_t)kc * p.N * 32, &tmF32, bar_in, 2 * p.inner + h * p.d + kc * 16, 0, 0, b);
            }
            mb_expect(bar_k, (uint32_t)(p.N * 128));
            tma4(K128, &tmF128, bar_k, p.inner + h * p.d, 0, 0, b);
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc1 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.N >> 3) << 17) | ((128u >> 4) << 24);
            const uint32_t idesc2 = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((64u >> 3) << 17) | ((128u >> 4) << 24);
            mb_wait(bar_in, 0);
            fence_after();
            for (int kc = 0; kc < p.kch; ++kc)
                mma_bf16(tmem_base, mdesc(s32(Qs) + (uint32_t)kc * 4096u, 16u, 256u, 6u),
                         mdesc(s32(K32) + (uint32_t)(kc * p.N * 32), 16u, 256u, 6u), idesc1, kc > 0 ? 1u : 0u);
            for (int kc = 0; kc < p.kch; ++kc)
                mma_bf16(tmem_base + 256u, mdesc(s32(Gs) + (uint32_t)kc * 4096u, 16u, 256u, 6u),
                         mdesc(s32(V32) + (uint32_t)(kc * p.N * 32), 16u, 256u, 6u), idesc1, kc > 0 ? 1u : 0u);
            mma_commit(bar_s);
            mb_wait(bar_k, 0);
            mb_wait(bar_ds, 0);
            fence_after();
            for (int kc = 0; kc < p.N / 16; ++kc)
                mma_bf16(tmem_base, mdesc(s32(Ss) + (uint32_t)kc * 4096u, 16u, 256u, 6u),
                         mdesc(s32(K128) + (uint32_t)(kc * 16 * 128), (uint32_t)(p.N * 128), 1024u, 2u), idesc2, kc > 0 ? 1u : 0u);
            mma_commit(bar_o);
        }
    } else {
        const int qd = warp & 3, row = qd * 32 + lane;
        const int q = qt * p.tok_t + row;
        const bool valid = row < p.tok_t && q < p.N;
        const int qq = valid ? q : 0;
        const int y = qq / p.W, x = qq - y * p.W;
        // D = dO . O for this query (bf16 token rows of `dout` / `out`), lse of the forward
        float D = 0.f, L = 0.f;
        if (valid) {
            const bf16* go = p.dout.at<bf16>(b, y, x, h * p.d);
            const bf16* oo = p.out.at<bf16>(b, y, x, h * p.d);
            for (int c = 0; c < p.d; c += 8) {
                const uint4 a = *reinterpret_cast<const uint4*>(go + c), o = *reinterpret_cast<const uint4*>(oo + c);
                const __nv_bfloat162* ha = reinterpret_cast<const __nv_bfloat162*>(&a);
                const __nv_bfloat162* ho = reinterpret_cast<const __nv_bfloat162*>(&o);
#pragma unroll
                for (int i = 0; i < 4; ++i) { const float2 fa = __bfloat1622float2(ha[i]), fo = __bfloat1622float2(ho[i]); D = fmaf(fa.x, fo.x, fmaf(fa.y, fo.y, D)); }
            }
            L = p.lse[((size_t)b * p.heads + h) * p.N + q];
            p.Dbuf[((size_t)b * p.heads + h) * p.N + q] = D;
        }
        const float Lb = L * 1.4426950408889634f;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(qd * 32) << 16);
        const uint32_t srow = s32(Ss) + (uint32_t)row * 32u, sw = (uint32_t)((row >> 2) & 1) << 4;
        mb_wait(bar_s, 0);
        fence_after();
        for (int c0 = 0; c0 < p.N; c0 += 16) {
            uint32_t rs[16], rp[16];
            tm_ld16(lane_addr + (uint32_t)c0, rs);
            tm_ld16(lane_addr + 256u + (uint32_t)c0, rp);
            tm_ld_wait();
            float e[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const float pij = exp2f(fmaf(__uint_as_float(rs[i]), p.scale_log2e, -Lb));
                e[i] = valid ? pij * (__uint_as_float(rp[i]) - D) : 0.f;
            }
            store_chunk_sw32(srow + (uint32_t)(c0 >> 4) * 4096u, sw, e);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        fence_before();
        mb_arrive(bar_ds);
        mb_wait(bar_o, 0);
        fence_after();
        bf16* drow = p.dqkv.at<bf16>(b, y, x, h * p.d);
        for (int c0 = 0; c0 < p.d; c0 += 16) {
            uint32_t r[16];
            tm_ld16(lane_addr + (uint32_t)c0, r);
            tm_ld_wait();
            if (valid) store_row16(drow + c0, r, p.scale);
        }
        fence_before();
    }
    __syncthreads();
    if (warp == 1) { fence_after(); tm_dealloc(tmem_base, 512u); }
}

// regions: o0 K tile [kch][128][32], o1 V tile [kch][128][32] (o0 doubles as the lse / D arrays once S^T, dP^T exist),
//          o2 Q32 [kch][N][32] then Q128 [N][128], o3 dO32 [kch][N][32] then dO128 [N][128], o4 P^T [N/16][128][32], o5 dS^T likewise
__global__ void __launch_bounds__(ATC_THREADS, 1) attn_bwd_dkv_tc_kernel(const __grid_constant__ CUtensorMap tmKt, const __grid_constant__ CUtensorMap tmQ32,
                                                                          const __grid_constant__ CUtensorMap tmG32, const __grid_constant__ CUtensorMap tmQ128,
                                                                          const __grid_constant__ CUtensorMap tmG128, AtbP p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t *Kt = smem + p.o0, *Vt = smem + p.o1, *Qr = smem + p.o2, *Gr = smem + p.o3, *Pt = smem + p.o4, *St = smem + p.o5;
    uint64_t* bars = (uint64_t*)(St + (size_t)(p.N / 16) * 4096);
    uint64_t *bar_in = bars, *bar_in2 = bars + 1, *bar_s = bars + 2, *bar_p = bars + 3, *bar_o = bars + 4;
    uint32_t* tmem_slot = (uint32_t*)(bars + 5);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int kt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmKt) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmQ32) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmG32) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmQ128) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmG128) : "memory");
        mb_init(bar_in, 1); mb_init(bar_in2, 1); mb_init(bar_s, 1); mb_init(bar_p, 128); mb_init(bar_o, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tm_alloc(tmem_slot, 512u);
    fence_before();
    __syncthreads();
    fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (warp == 0) {
        if (lane == 0) {
            mb_expect(bar_in, (uint32_t)(p.kch * (2 * p.tok_t + 2 * p.N) * 32));
            for (int kc = 0; kc < p.kch; ++kc) {
                tma4(Kt + (size_t)kc * 4096, &tmKt, bar_in, p.inner + h * p.d + kc * 16, 0, kt * p.rows_t, b);
                tma4(Vt + (size_t)kc * 4096, &tmKt, bar_in, 2 * p.inner + h * p.d + kc * 16, 0, kt * p.rows_t, b);
                tma4(Qr + (size_t)kc * p.N * 32, &tmQ32, bar_in, h * p.d + kc * 16, 0, 0, b);
                tma4(Gr + (size_t)kc * p.N * 32, &tmG32, bar_in, h * p.d + kc * 16, 0, 0, b);
            }
            // the MN-major copies of Q and dO replace the K-major ones once S^T and dP^T are complete
            mb_wait(bar_s, 0);
            mb_expect(bar_in2, (uint32_t)(2 * p.N * 128));
            tma4(Qr, &tmQ128, bar_in2, h * p.d, 0, 0, b);
            tma4(Gr, &tmG128, bar_in2, h * p.d, 0, 0, b);
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc1 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.N >> 3) << 17) | ((128u >> 4) << 24);
            const uint32_t idesc2 = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((64u >> 3) << 17) | ((128u >> 4) << 24);
            mb_wait(bar_in, 0);
            fence_after();
            for (int kc = 0; kc < p.kch; ++kc)
                mma_bf16(tmem_base, mdesc(s32(Kt) + (uint32_t)kc * 4096u, 16u, 256u, 6u),
                         mdesc(s32(Qr) + (uint32_t)(kc * p.N * 32), 16u, 256u, 6u), idesc1, kc > 0 ? 1u : 0u);
            for (int kc = 0; kc < p.kch; ++kc)
                mma_bf16(tmem_base + 256u, mdesc(s32(Vt) + (uint32_t)kc * 4096u, 16u, 256u, 6u),
                         mdesc(s32(Gr) + (uint32_t)(kc * p.N * 32), 16u, 256u, 6u), idesc1, kc > 0 ? 1u : 0u);
            mma_commit(bar_s);
            mb_wait(bar_in2, 0);
            mb_wait(bar_p, 0);
            fence_after();
            for (int kc = 0; kc < p.N / 16; ++kc)        // dV = P^T dO  -> TMEM columns 0..63
                mma_bf16(tmem_base, mdesc(s32(Pt) + (uint32_t)kc * 4096u, 16u, 256u, 6u),
                         mdesc(s32(Gr) + (uint32_t)(kc * 16 * 128), (uint32_t)(p.N * 128), 1024u, 2u), idesc2, kc > 0 ? 1u : 0u);
            for (int kc = 0; kc < p.N / 16; ++kc)        // dK = dS^T Q -> TMEM columns 64..127
                mma_bf16(tmem_base + 64u, mdesc(s32(St) + (uint32_t)kc * 4096u, 16u, 256u, 6u),
                         mdesc(s32(Qr) + (uint32_t)(kc * 16 * 128), (uint32_t)(p.N * 128), 1024u, 2u), idesc2, kc > 0 ? 1u : 0u);
            mma_commit(bar_o);
        }
    } else {
        const int qd = warp & 3, row = qd * 32 + lane;
        const int j = kt * p.tok_t + row;
        const bool valid = row < p.tok_t && j < p.N;
        const int jj = valid ? j : 0;
        const int y = jj / p.W, x = jj - y * p.W;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(qd * 32) << 16);
        const uint32_t prow = s32(Pt) + (uint32_t)row * 32u, srow = s32(St) + (uint32_t)row * 32u, sw = (uint32_t)((row >> 2) & 1) << 4;
        mb_wait(bar_s, 0);                                // S^T, dP^T complete: the K / V tiles are dead -> per-query lse, D go there
        fence_after();
        float* Ls = reinterpret_cast<float*>(Kt);
        float* Ds = Ls + p.N;
        for (int i = threadIdx.x - 64; i < p.N; i += 128) {
            Ls[i] = p.lse[((size_t)b * p.heads + h) * p.N + i] * 1.4426950408889634f;
            Ds[i] = p.Dbuf[((size_t)b * p.heads + h) * p.N + i];
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
        for (int c0 = 0; c0 < p.N; c0 += 16) {
            uint32_t rs[16], rp[16];
            tm_ld16(lane_addr + (uint32_t)c0, rs);
            tm_ld16(lane_addr + 256u + (uint32_t)c0, rp);
            tm_ld_wait();
            float e[16], f[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const float pij = valid ? exp2f(fmaf(__uint_as_float(rs[i]), p.scale_log2e, -Ls[c0 + i])) : 0.f;
                e[i] = pij;
                f[i] = valid ? pij * (__uint_as_float(rp[i]) - Ds[c0 + i]) : 0.f;
            }
            store_chunk_sw32(prow + (uint32_t)(c0 >> 4) * 4096u, sw, e);
            store_chunk_sw32(srow + (uint32_t)(c0 >> 4) * 4096u, sw, f);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        fence_before();
        mb_arrive(bar_p);
        mb_wait(bar_o, 0);
        fence_after();
        bf16* krow = p.dqkv.at<bf16>(b, y, x, p.inner + h * p.d);
        bf16* vrow = p.dqkv.at<bf16>(b, y, x, 2 * p.inner + h * p.d);
        for (int c0 = 0; c0 < p.d; c0 += 16) {
            uint32_t rv[16], rk[16];
            tm_ld16(lane_addr + (uint32_t)c0, rv);
            tm_ld16(lane_addr + 64u + (uint32_t)c0, rk);
            tm_ld_wait();
            if (valid) { store_row16(vrow + c0, rv, 1.0f); store_row16(krow + c0, rk, p.scale); }
        }
        fence_before();
    }
    __syncthreads();
    if (warp == 1) { fence_after(); tm_dealloc(tmem_base, 512u); }
}

}  // namespace

// N = H*W <= 256 keys (a multiple of 16), head_dim 32 / 64 (V is fetched as a 64-channel box: with head_dim 32 the upper 32
// output columns are the next head's and are ignored), query tiles of whole image rows.
int attn_tc_supported(const ddpm_tensor* qkv, const ddpm_tensor* out, int heads, int d, int dtype) {
    if (dtype != DDPM_BF16 || (d != 32 && d != 64)) return 0;
    const int N = qkv->H * qkv->W;
    if (N > 256 || N % 16 || qkv->W > 256 || qkv->H > 256) return 0;
    if (N > 128 && (128 % qkv->W || N % 128)) return 0;
    if (qkv->halo != 1 && qkv->halo != 0) return 0;
    if (qkv->pitch % 8 || out->pitch % 8 || ((uintptr_t)qkv->ptr & 15) || ((uintptr_t)out->ptr & 15)) return 0;
    if ((heads * d) % 8) return 0;
    return 1;
}

int attn_tc_launch(const ddpm_tensor* qkv, const ddpm_tensor* out, int heads, int d, float* lse, cudaStream_t st) {
    AtcP p;
    p.out = TV(*out); p.lse = lse; p.heads = heads; p.d = d; p.inner = heads * d;
    p.N = qkv->H * qkv->W; p.NK = p.N; p.W = qkv->W;
    p.tok_q = p.N < 128 ? p.N : 128; p.rows_q = p.tok_q / qkv->W;
    p.kch = d / 16;
    p.scale = 1.0f / sqrtf((float)d); p.scale_log2e = p.scale * 1.4426950408889634f;
    p.q_off = 0;
    p.k_off = p.kch * 4096;
    p.v_off = (p.k_off + p.kch * p.NK * 32 + 1023) & ~1023;
    p.p_off = (p.v_off + p.NK * 128 + 1023) & ~1023;
    const size_t smem = (size_t)p.p_off + (size_t)(p.NK / 16) * 4096 + 8 * 5 + 16 + 1024;
    CUtensorMap tmQ, tmK, tmV;
    {
        const int Hp = qkv->H + 2 * qkv->halo, Wp = qkv->W + 2 * qkv->halo;
        char* base = (char*)qkv->ptr + ((size_t)qkv->halo * Wp + qkv->halo) * qkv->pitch * 2;
        const uint64_t dims[4] = {(uint64_t)qkv->C, (uint64_t)qkv->W, (uint64_t)qkv->H, (uint64_t)qkv->N};
        const uint64_t strides[3] = {(uint64_t)qkv->pitch * 2, (uint64_t)Wp * qkv->pitch * 2, (uint64_t)Hp * Wp * qkv->pitch * 2};
        const uint32_t bq[4] = {16u, (uint32_t)qkv->W, (uint32_t)p.rows_q, 1u};
        const uint32_t bk[4] = {16u, (uint32_t)qkv->W, (uint32_t)qkv->H, 1u};
        const uint32_t bv[4] = {64u, (uint32_t)qkv->W, (uint32_t)qkv->H, 1u};
        int rc = ddpm_encode_tiled_bf16(&tmQ, base, 4, dims, strides, bq, 32); if (rc) return rc;
        rc = ddpm_encode_tiled_bf16(&tmK, base, 4, dims, strides, bk, 32); if (rc) return rc;
        rc = ddpm_encode_tiled_bf16(&tmV, base, 4, dims, strides, bv, 128); if (rc) return rc;
    }
    static size_t configured = 0;
    if (smem > configured) {
        CUDA_TRY(cudaFuncSetAttribute(attn_fwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = smem;
    }
    dim3 grid((p.N + p.tok_q - 1) / p.tok_q, heads, qkv->N);
    CUDA_TRY(launch_kernel(attn_fwd_tc_kernel, grid, dim3(ATC_THREADS), smem, st, tmQ, tmK, tmV, p));
    LAUNCH_OK();
    return 0;
}

static int atc_maps(const ddpm_tensor* t, int rows_tile, CUtensorMap* tile32, CUtensorMap* full32, CUtensorMap* full128) {
    const int Hp = t->H + 2 * t->halo, Wp = t->W + 2 * t->halo;
    char* base = (char*)t->ptr + ((size_t)t->halo * Wp + t->halo) * t->pitch * 2;
    const uint64_t dims[4] = {(uint64_t)t->C, (uint64_t)t->W, (uint64_t)t->H, (uint64_t)t->N};
    const uint64_t strides[3] = {(uint64_t)t->pitch * 2, (uint64_t)Wp * t->pitch * 2, (uint64_t)Hp * Wp * t->pitch * 2};
    const uint32_t bt[4] = {16u, (uint32_t)t->W, (uint32_t)rows_tile, 1u};
    const uint32_t bf[4] = {16u, (uint32_t)t->W, (uint32_t)t->H, 1u};
    const uint32_t bw[4] = {64u, (uint32_t)t->W, (uint32_t)t->H, 1u};
    int rc = 0;
    if (tile32) { rc = ddpm_encode_tiled_bf16(tile32, base, 4, dims, strides, bt, 32); if (rc) return rc; }
    if (full32) { rc = ddpm_encode_tiled_bf16(full32, base, 4, dims, strides, bf, 32); if (rc) return rc; }
    if (full128) { rc = ddpm_encode_tiled_bf16(full128, base, 4, dims, strides, bw, 128); if (rc) return rc; }
    return 0;
}

// floats of scratch the tensor-core backward needs (D = dO . O per query) -- 0 when the shape is not eligible
int64_t attn_tc_bwd_scratch_floats(const ddpm_tensor* qkv, const ddpm_tensor* out, int heads, int d, int dtype) {
    if (!attn_tc_supported(qkv, out, heads, d, dtype)) return 0;
    return (int64_t)qkv->N * heads * qkv->H * qkv->W;
}

int attn_tc_bwd_launch(const ddpm_tensor* qkv, const ddpm_tensor* out, const ddpm_tensor* dout, const float* lse,
                       const ddpm_tensor* dqkv, int heads, int d, float* scratch, cudaStream_t st) {
    AtbP p;
    p.out = TV(*out); p.dout = TV(*dout); p.dqkv = TV(*dqkv); p.lse = lse; p.Dbuf = scratch;
    p.heads = heads; p.d = d; p.inner = heads * d; p.N = qkv->H * qkv->W; p.W = qkv->W;
    p.tok_t = p.N < 128 ? p.N : 128; p.rows_t = p.tok_t / qkv->W; p.kch = d / 16;
    p.scale = 1.0f / sqrtf((float)d); p.scale_log2e = p.scale * 1.4426950408889634f;
    const int A1 = p.kch * 4096, AN = (p.kch * p.N * 32 + 1023) & ~1023, W128 = (p.N * 128 + 1023) & ~1023, CH = (p.N / 16) * 4096;
    CUtensorMap qT, qF32, qF128, gT, gF32, gF128;
    int rc = atc_maps(qkv, p.rows_t, &qT, &qF32, &qF128); if (rc) return rc;
    rc = atc_maps(dout, p.rows_t, &gT, &gF32, &gF128); if (rc) return rc;
    dim3 grid((p.N + p.tok_t - 1) / p.tok_t, heads, qkv->N);
    {   // dq: Q, dO, K32, V32, K128, dS
        p.o0 = 0; p.o1 = A1; p.o2 = 2 * A1; p.o3 = p.o2 + AN; p.o4 = p.o3 + AN; p.o5 = p.o4 + W128;
        const size_t smem = (size_t)p.o5 + CH + 8 * 5 + 16 + 1024;
        static size_t configured = 0;
        if (smem > configured) { CUDA_TRY(cudaFuncSetAttribute(attn_bwd_dq_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); configured = smem; }
        CUDA_TRY(launch_kernel(attn_bwd_dq_tc_kernel, grid, dim3(ATC_THREADS), smem, st, qT, gT, qF32, qF128, p));
        LAUNCH_OK();
    }
    {   // dkv: K tile, V tile, Q32 -> Q128, dO32 -> dO128, P^T, dS^T
        const int R = AN > W128 ? AN : W128;
        p.o0 = 0; p.o1 = A1; p.o2 = 2 * A1; p.o3 = p.o2 + R; p.o4 = p.o3 + R; p.o5 = p.o4 + CH;
        const size_t smem = (size_t)p.o5 + CH + 8 * 5 + 16 + 1024;
        static size_t configured = 0;
        if (smem > configured) { CUDA_TRY(cudaFuncSetAttribute(attn_bwd_dkv_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); configured = smem; }
        CUDA_TRY(launch_kernel(attn_bwd_dkv_tc_kernel, grid, dim3(ATC_THREADS), smem, st, qT, qF32, gF32, qF128, gF128, p));
        LAUNCH_OK();
    }
    return 0;
}
