// tcgen05 / TMEM implicit-GEMM convolution for sm_100a (bf16 in, fp32 accumulate in tensor memory).
//
// "Shift-GEMM" over the padded NHWC layout.  Activations carry a zero halo, so with
// Q = (n*Hp + yp)*Wp + xp the padded-linear pixel index, a 3x3/s1/p1 convolution is
//     out[Q][co] = sum_{ky,kx} sum_ci  A[Q + (ky-1)*Wp + (kx-1)][ci] * W[co][ky][kx][ci]
// for every interior Q: each filter tap is a constant ROW SHIFT of the same [pixels x channels]
// matrix.  A CTA therefore stages one halo'd patch of 128*MT + 2*Wp + 2 pixel rows per 16-channel
// K-chunk ONCE (TMA, zero-filled outside the tensor) and issues all nine taps as tcgen05.mma
// instructions whose shared-memory descriptors differ only in their start address -- the 9x im2col
// re-read of the activation never happens (neither from HBM nor from L2).  Outputs computed at halo
// positions are discarded by the epilogue, which keeps the output halo zero.
//
// Replaces cuDNN behind nn.Conv2d 3x3 s1 / 1x1 (unet_backbone.py:22,32,35,60; attention.py:53-54)
// for fprop and, with flipped/transposed weights, dgrad.
#include "common.cuh"
#include <cuda.h>
#include <type_traits>
#include <cudaTypedefs.h>

#define TC_THREADS 192
#define KC 16                 // channels per K-chunk (one UMMA K step for bf16)

static int sm_count();
// path-forcing flags of ddpm_set_tc_mode (mode >> 4, see ddpm_b200.h), read by the launch planners below
static int g_tc_exp = 0;
extern "C" int ddpm_set_tc_mode(int mode, int base_offset) {
    if ((mode & 15) != 1 || base_offset != 0 || ((mode >> 4) & ~(32 | 64 | 128 | 1024))) return DDPM_E_ARG;
    g_tc_exp = mode >> 4;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(smem_u32(dst)), "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptors (cute::UMMA::SmemDescriptor bit layout: start address >> 4, LBO >> 4 at bit 16,
// SBO >> 4 at bit 32, version 1 at bit 46, layout at bit 61).  The base offset (bits 49-51) stays 0: the swizzle is a
// pure function of the shared-memory address, so row-shifted descriptors need no correction (measured on B200).
// The MMA-issuing thread is a single lane: every integer instruction between two tcgen05.mma costs
// ~5 cycles of dependent latency, and a loop that rebuilds both 64-bit descriptors (shifts, masks,
// tap / 3, tap % 3) per MMA was measured at 137-230 cycles per MMA -- above the 48-128 cycle tensor
// floor, i.e. the kernel was ISSUE-bound, independent of N (profiles/r1_conv_issue_bound.txt).
// Descriptors are therefore split into a constant high word and a low word (address | LBO) that
// advances by plain 32-bit adds.
__device__ __forceinline__ uint64_t desc_pack(uint32_t lo, uint32_t hi) {
    uint64_t d; asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "r"(lo), "r"(hi)); return d;
}
__device__ __forceinline__ uint32_t desc_hi(uint32_t sbo_bytes, uint32_t layout) {
    return ((sbo_bytes >> 4) & 0x3FFF) | (1u << 14) | ((layout & 7) << 29);
}
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr, uint32_t lbo_bytes) {
    return ((saddr >> 4) & 0x3FFF) | (((lbo_bytes >> 4) & 0x3FFF) << 16);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static PFN_cuTensorMapEncodeTiled_v12000 g_encode = nullptr;
static int get_encode() {
    if (g_encode) return 0;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) return 801;   // cudaErrorNotSupported
    g_encode = (PFN_cuTensorMapEncodeTiled_v12000)fn;
    return 0;
}

static int encode(CUtensorMap* m, void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                  const uint32_t* box, CUtensorMapSwizzle sw) {
    cuuint64_t gd[5]; cuuint64_t gs[4]; cuuint32_t bx[5]; cuuint32_t es[5];
    for (int i = 0; i < rank; ++i) { gd[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
    for (int i = 0; i < rank - 1; ++i) gs[i] = strides_bytes[i];
    CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, base, gd, gs, bx, es,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : 1;   // cudaErrorInvalidValue
}

// shared with attn_tc.cu: bf16 tiled tensor map, swizzle_bytes in {0, 32, 64, 128}
int ddpm_encode_tiled_bf16(CUtensorMap* m, void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                           const uint32_t* box, int swizzle_bytes) {
    int rc = get_encode(); if (rc) return rc;
    const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                : swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
    return encode(m, base, rank, dims, strides_bytes, box, sw);
}

static int pick_nt(int Cout) {
    if (Cout <= 256) return Cout;
    for (int nt = 256; nt >= 64; nt -= 16) if (Cout % nt == 0) return nt;
    return 0;
}

int conv_tc_supported(const ddpm_conv_args* a) {
    const bool up = a->mode == DDPM_CONV_UP2X_PHASE;
    if (a->dtype != DDPM_BF16 || (a->mode != DDPM_CONV_NORMAL && !up) || a->a_silu || a->z.ptr) return 0;
    if (up) { if (a->KH != 2 || a->KW != 2 || a->stride != 1 || a->res.ptr || a->in2.ptr || (a->epi & DDPM_EPI_ACCUM)) return 0; }
    else if (!((a->KH == 3 && a->KW == 3 && a->pad == 1) || (a->KH == 1 && a->KW == 1 && a->pad == 0))) return 0;
    const ddpm_tensor &in = a->in, &out = a->out;
    if (in.halo != 1 || out.halo != 1 || in.N != out.N) return 0;
    if (up) { if (out.H != 2 * in.H || out.W != 2 * in.W) return 0; }
    else if (a->stride == 1) { if (in.H != out.H || in.W != out.W) return 0; }
    else if (a->stride == 2) { if (a->KH != 3 || (in.H & 1) || (in.W & 1) || out.H * 2 != in.H || out.W * 2 != in.W) return 0; }
    else return 0;
    if (in.C % 16 || out.C % 16 || in.pitch % 8 || out.pitch % 8) return 0;
    if (((uintptr_t)in.ptr & 15) || ((uintptr_t)out.ptr & 15) || ((uintptr_t)a->w & 15)) return 0;
    if (a->res.ptr && (a->res.halo != 1 || a->res.pitch % 8 || ((uintptr_t)a->res.ptr & 15))) return 0;
    if (pick_nt(out.C) == 0) return 0;
    if (in.W + 2 > 300) return 0;         // patch would not fit the A ring (large images: later round)
    if (a->in2.ptr) {                     // fused 1x1 second operand: persistent pair kernel, 3x3 stride-1 main conv only
        const ddpm_tensor& i2 = a->in2;
        if (a->KH != 3 || a->stride != 1 || (a->epi & DDPM_EPI_DSILU)) return 0;
        if (i2.halo != 1 || i2.C % 16 || i2.pitch % 8 || ((uintptr_t)i2.ptr & 15) || ((uintptr_t)a->w2 & 15)) return 0;
    }
    return 1;
}

// ================================================================================================
// persistent CTA-PAIR kernel (cta_group::2), TMEM double-buffered
//
// Why (ncu, profiles/r1_ncu_prof_conv_tc_192_64.txt): a kernel with one 128/256-pixel tile per CTA re-fetches the
// whole 9-tap weight slab for every tile -- 87 % of its 3.3 GB of L2->SM traffic at 192->192@64 -- and two
// co-resident CTAs fall into lock-step, so the tensor pipe is active 33 % of the time.  Here
//   * two CTAs of a cluster (one TPC) issue M=256 MMAs: each CTA stages its own 128*MT pixel rows (A) but
//     only HALF of the weight tile (B); the tensor cores of both SMs read both halves -> B traffic / 2;
//   * one CTA per SM, ~200 KB operand ring (6-8 K-chunks in flight, covers the TMA round trip);
//   * the CTA pair is persistent and walks (pixel tile, channel tile) items; accumulators are double
//     buffered in TMEM (2 x MT*NT columns), so the epilogue of item i overlaps the MMAs of item i+1 and
//     the producer prefetches across item boundaries.
// Barrier protocol (same smem offsets in both CTAs):
//   full[s]   (leader)  : 1 arrive.expect_tx(bytes of BOTH CTAs); both CTAs' TMA loads complete_tx on it
//   empty[s]  (each CTA): tcgen05.commit.cta_group::2 multicast to both CTAs
//   tfull[b]  (each CTA): commit multicast after the item's last MMA -> the CTA's own epilogue warps
//   tempty[b] (leader)  : 4 epilogue warps x 2 CTAs arrive (remote arrive from the peer)
// ================================================================================================
#define TC2_THREADS 320          // warp 0 TMA, warp 1 MMA issue, warps 2..9 epilogue (two per TMEM lane quarter)
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
    uint32_t r; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank)); return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    // relaxed: the arrive only publishes "my tcgen05.ld of this accumulator buffer are done" (ordered by
    // tcgen05.fence::before_thread_sync); a release here would also wait for the epilogue's global stores
    // to drain (ncu: MEMBAR + ERRBAR = 16 % of the stall samples) for no reason
    asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tma2_load_2d(void* dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(smem_u32(dst)), "l"(m), "r"(bar_cluster_addr), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma2_load_3d(void* dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 ::"r"(smem_u32(dst)), "l"(m), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma2_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma2_commit_mc(uint64_t* bar) {      // arrives on `bar` in BOTH CTAs of the pair
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}

// 256-bit global accesses (sm_100: LDG/STG.E.ENL2.256): one full 32-byte sector per lane and instruction.  The
// epilogue's rows are 192-384 B apart, so every lane touches its own sector anyway; with 16-byte accesses each
// sector was written (and, for residuals, read) in two halves by two instructions.
struct U8 { uint4 lo, hi; };
__device__ __forceinline__ void ldg256(const void* p, U8& v) {
    asm volatile("ld.global.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v.lo.x), "=r"(v.lo.y), "=r"(v.lo.z), "=r"(v.lo.w), "=r"(v.hi.x), "=r"(v.hi.y), "=r"(v.hi.z), "=r"(v.hi.w) : "l"(p));
}
__device__ __forceinline__ void stg256(void* p, const uint4& lo, const uint4& hi) {
    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 ::"l"(p), "r"(lo.x), "r"(lo.y), "r"(lo.z), "r"(lo.w), "r"(hi.x), "r"(hi.y), "r"(hi.z), "r"(hi.w) : "memory");
}

struct Tc2Params {
    TV out, res;
    const float* bias; const float* tbias; int tbias_pitch; int bias_n;
    int Cin, Cout, NT, n_tiles;   // NT: UMMA N (full tile, both halves); each CTA stages NT/2 weight rows per tap
    int taps;                     // 9 or 1
    int Hp, Wp, H, W, Qtot;
    int P, seg;                   // patch rows per K-chunk, TMA box height
    int KS;                       // K-chunks per ring stage (1 for 3x3, up to 4 for 1x1)
    int S;                        // ring depth
    int a_chunk_bytes, b_chunk_bytes, stage_bytes;
    int pix_tiles, items;
    int has_res, accum, sub;
    int vec_bias, vec_tbias;      // 16-byte aligned -> float4 loads in the epilogue
    int v256;                     // out (and res) rows are 32-byte aligned -> 256-bit loads / stores
    int b_res;                    // 1: this CTA's half of the weight tile (all K-chunks, all taps) stays resident in shared
                                  //    memory -- loaded once, with the first item's stages -- and only A patches stream
    int up, py, px;               // DDPM_CONV_UP2X_PHASE: 2x2 taps at rows y+ty+py-1 / columns x+tx+px-1 of the low-resolution input,
                                  //    results stored at (2y+py, 2x+px) of the full-resolution output
    int KCH2;                     // K-chunks of the fused 1x1 second operand (0: none): they follow the 3x3 chunks of every
    int b2_chunk_bytes;           //    item, load their patch through tmA2 / their one-tap weight slab through tmB2 and
                                  //    issue only the centre tap
};

// FUSED2: the 1x1 second operand (ddpm_conv_args.in2).  A template parameter, not a run-time branch: the extra stage kind
// in the producer and MMA-issue loops cost 3-4 % on EVERY convolution when it was one (A/B of three builds on one box,
// 96->96@64: 67.9 -> 70.0 us) -- the issue loop is that tight.
template <int MT, int TAPS, bool FUSED2>
__global__ void __launch_bounds__(TC2_THREADS, 1) conv_tc2_kernel(const __grid_constant__ CUtensorMap tmA,
                                                                  const __grid_constant__ CUtensorMap tmB,
                                                                  const __grid_constant__ CUtensorMap tmA2,
                                                                  const __grid_constant__ CUtensorMap tmB2, Tc2Params p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* ring = smem;
    uint8_t* bres = ring + (size_t)p.S * p.stage_bytes;                                   // resident weights (b_res only)
    uint64_t* bars = (uint64_t*)(bres + (p.b_res ? (size_t)(p.Cin / KC) * p.b_chunk_bytes + (FUSED2 ? (size_t)p.KCH2 * p.b2_chunk_bytes : 0) : 0));
    uint64_t* full = bars;            uint64_t* empty = full + p.S;
    uint64_t* tfull = empty + p.S;    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_slot = (uint32_t*)(tempty + 2);
    float* sbias = (float*)(tmem_slot + 4);              // [Cout] bias staged once per CTA (16-byte aligned: the barrier block is)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
    const int KCH = p.Cin / KC;
    const int KCH2 = FUSED2 ? p.KCH2 : 0;
    const int NST = (KCH + p.KS - 1) / p.KS + KCH2;     // ring stages per item (KS = 1 whenever a second operand is fused)
    const int halo_rows = (p.taps > 1) ? p.Wp + 1 : 0;
    const int tile_rows = 128 * MT;
    const int cols_per_buf = MT * p.NT;

    if (threadIdx.x == 0) {
        // descriptor fetch (128 B each from the parameter bank) overlaps barrier set-up / TMEM allocation / cluster sync
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
        if (FUSED2) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA2) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB2) : "memory");
        }
        for (int i = 0; i < p.S; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], 16); }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc2(tmem_slot, 512u);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                  // peer's barriers are initialised before anyone signals them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // The bias vector is read by every epilogue trip; as __ldg float4 loads after the accumulator wait it cost ~25 % of the
    // epilogue at 96 channels (measured when the time bias absorbed conv1's bias).  Stage it in shared memory once.
    if (p.bias && warp >= 2 && warp < 10) {
        for (int i = threadIdx.x - 64; i < p.Cout; i += TC2_THREADS - 64) sbias[i] = i < p.bias_n ? __ldg(p.bias + i) : 0.f;
        asm volatile("bar.sync 1, %0;" ::"n"(TC2_THREADS - 64) : "memory");      // epilogue warps only
    }

    if (warp == 0) {
        // ===================================================================== TMA producer (both CTAs)
        if (lane == 0) {
            uint32_t g = 0;                              // global stage counter (continues across items)
            for (int it = pair; it < p.items; it += npairs) {
                const int pt = it / p.n_tiles, ntile = it - pt * p.n_tiles;
                const int Q0 = pt * (2 * tile_rows) + (int)rank * tile_rows;
                const int nrow0 = ntile * p.NT + (int)rank * (p.NT / 2);
                for (int st = 0; st < NST; ++st, ++g) {
                    const int s = g % p.S; const uint32_t ph = (g / p.S) & 1;
                    mbar_wait(&empty[s], ph ^ 1);
                    const bool second = FUSED2 && st >= NST - KCH2;               // a chunk of the fused 1x1 operand
                    const int kc0 = second ? st - (NST - KCH2) : st * p.KS, nk = second ? 1 : min(p.KS, KCH - kc0);
                    const uint32_t fbar = mapa_u32(smem_u32(&full[s]), 0);
                    const bool loadB = !(p.b_res && it != pair);                 // resident weights arrive with the first item only
                    const int bbytes = second ? p.b2_chunk_bytes : p.b_chunk_bytes;
                    const uint32_t tx = (uint32_t)(2 * nk * (p.P * 32 + (loadB ? bbytes : 0)));
                    if (leader) mbar_expect_tx(&full[s], tx);
                    uint8_t* sbase = ring + (size_t)s * p.stage_bytes;
                    const CUtensorMap* mA = second ? &tmA2 : &tmA;
                    const CUtensorMap* mB = second ? &tmB2 : &tmB;
                    for (int k = 0; k < nk; ++k) {
                        uint8_t* adst = sbase + (size_t)k * (p.a_chunk_bytes + (p.b_res ? 0 : p.b_chunk_bytes));
                        uint8_t* bdst = !p.b_res ? adst + p.a_chunk_bytes
                                      : (second ? bres + (size_t)KCH * p.b_chunk_bytes + (size_t)kc0 * p.b2_chunk_bytes
                                                : bres + (size_t)(kc0 + k) * p.b_chunk_bytes);
                        const int row0 = Q0 - halo_rows;
                        for (int r = 0; r < p.P; r += p.seg)
                            tma2_load_2d(adst + (size_t)r * 32, mA, fbar, (kc0 + k) * KC, row0 + r);
                        if (loadB) tma2_load_3d(bdst, mB, fbar, (kc0 + k) * KC, nrow0, 0);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===================================================================== MMA issuer (leader CTA only)
        // the whole warp runs the loop (warp-uniform control flow keeps descriptors in uniform registers);
        // one elected lane issues the tcgen05 instructions
        if (leader) {
            const bool el = elect_one();
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.NT >> 3) << 17) | ((256u >> 4) << 24);
            const uint32_t hi = desc_hi(256u, 6u);                       // SBO 256 B, SWIZZLE_32B
            uint32_t tapoff[TAPS];                                       // A row shift of each tap, in 16-byte units
#pragma unroll
            for (int tap = 0; tap < TAPS; ++tap)
                tapoff[tap] = TAPS == 9 ? (uint32_t)(((tap / 3) * p.Wp + (tap % 3)) * 2)
                            : TAPS == 4 ? (uint32_t)((((tap >> 1) + p.py) * p.Wp + ((tap & 1) + p.px)) * 2) : 0u;
            const uint32_t b_tap = (uint32_t)p.NT;                       // (NT/2 rows * 32 B) >> 4
            const uint32_t chunk16 = (uint32_t)((p.a_chunk_bytes + (p.b_res ? 0 : p.b_chunk_bytes)) >> 4), a16 = (uint32_t)(p.a_chunk_bytes >> 4);
            const uint32_t ring_lo = desc_lo(smem_u32(ring), 16u), stage16 = (uint32_t)(p.stage_bytes >> 4);
            const uint32_t bres_lo = desc_lo(smem_u32(bres), 16u), bchunk16 = (uint32_t)(p.b_chunk_bytes >> 4);
            uint32_t g = 0, j = 0;
            for (int it = pair; it < p.items; it += npairs, ++j) {
                const uint32_t buf = j & 1, bph = (j >> 1) & 1;
                mbar_wait(&tempty[buf], bph ^ 1);        // both CTAs' epilogues have drained this accumulator buffer
                tc_fence_after();
                const uint32_t dbase = tmem_base + buf * (uint32_t)cols_per_buf;
                uint32_t acc = 0;
                for (int st = 0; st < NST; ++st, ++g) {
                    const uint32_t s = g % (uint32_t)p.S; const uint32_t ph = (g / (uint32_t)p.S) & 1;
                    mbar_wait(&full[s], ph);
                    tc_fence_after();
                    uint32_t a_lo = ring_lo + s * stage16;
                    if (FUSED2 && st >= NST - KCH2) {
                        // fused 1x1 operand: one MMA per M-tile, the patch's centre tap against the one-tap weight slab
                        const uint32_t kc2 = (uint32_t)(st - (NST - KCH2));
                        const uint32_t b_lo = p.b_res ? bres_lo + (uint32_t)KCH * bchunk16 + kc2 * (uint32_t)(p.b2_chunk_bytes >> 4) : a_lo + a16;
                        const uint64_t bdesc = desc_pack(b_lo, hi);
#pragma unroll
                        for (int mt = 0; mt < MT; ++mt) {
                            const uint64_t adesc = desc_pack(a_lo + tapoff[TAPS / 2] + (uint32_t)(mt * 256), hi);
                            if (el) umma2_bf16(dbase + (uint32_t)(mt * p.NT), adesc, bdesc, idesc, 1u);
                        }
                        if (el) umma2_commit_mc(&empty[s]);
                        __syncwarp();
                        continue;
                    }
                    const int nk = TAPS > 1 ? 1 : min(p.KS, KCH - st * p.KS);       // 3x3 / 2x2: one K-chunk per stage, always
                    for (int k = 0; k < nk; ++k, a_lo += chunk16) {
                        const uint32_t b_lo = p.b_res ? bres_lo + (uint32_t)((TAPS > 1 ? st : st * p.KS) + k) * bchunk16 : a_lo + a16;
#pragma unroll
                        for (int tap = 0; tap < TAPS; ++tap) {
                            const uint64_t bdesc = desc_pack(b_lo + (uint32_t)tap * b_tap, hi);
#pragma unroll
                            for (int mt = 0; mt < MT; ++mt) {
                                const uint64_t adesc = desc_pack(a_lo + tapoff[tap] + (uint32_t)(mt * 256), hi);
                                if (el) umma2_bf16(dbase + (uint32_t)(mt * p.NT), adesc, bdesc, idesc, tap == 0 ? acc : 1u);
                            }
                        }
                        acc = 1;
                    }
                    if (el) umma2_commit_mc(&empty[s]);
                    __syncwarp();
                }
                if (el) umma2_commit_mc(&tfull[buf]);
                __syncwarp();
            }
        }
    } else {
        // ===================================================================== epilogue (both CTAs)
        const int qd = warp & 3;                          // TMEM lane quarter this warp may read (warp id % 4)
        const int half = (warp - 2) >> 2;                 // the two warps of a quarter split the 16-column blocks
        const int nblk = p.NT >> 4;
        const int blk_lo = half ? (nblk + 1) / 2 : 0, blk_hi = half ? nblk : (nblk + 1) / 2;
        const int HpWp = p.Hp * p.Wp;
        const uint32_t tempty_leader0 = mapa_u32(smem_u32(&tempty[0]), 0);
        const uint32_t tempty_leader1 = mapa_u32(smem_u32(&tempty[1]), 0);
        uint32_t j = 0;
        for (int it = pair; it < p.items; it += npairs, ++j) {
            const uint32_t buf = j & 1, bph = (j >> 1) & 1;
            const int pt = it / p.n_tiles, ntile = it - pt * p.n_tiles;
            const int Q0 = pt * (2 * tile_rows) + (int)rank * tile_rows;
            const int n0 = ntile * p.NT;
            // Row addressing for this item is done BEFORE waiting for the accumulators, and the residual / accumulate
            // rows are prefetched into L2 while the MMAs are still running: the epilogue was latency-bound on
            // those reads (96->96@64: 75 us plain vs 140 us with a residual).
            bf16* orow_a[MT]; const bf16* rrow_a[MT]; const float* tb_a[MT];
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
                const int Q = Q0 + mt * 128 + qd * 32 + lane;
                bool valid = Q < p.Qtot;
                int n = 0, y = 0, x = 0;
                if (valid) {
                    n = Q / HpWp; int r = Q - n * HpWp; int yp = r / p.Wp; int xp = r - yp * p.Wp;
                    y = yp - 1; x = xp - 1;
                    valid = y >= 0 && y < p.H && x >= 0 && x < p.W;
                    if (p.sub) { valid = valid && ((y | x) & 1) == 0; y >>= 1; x >>= 1; }
                    if (p.up) { y = 2 * y + p.py; x = 2 * x + p.px; }
                }
                orow_a[mt] = valid ? p.out.at<bf16>(n, y, x, n0) : nullptr;
                rrow_a[mt] = (valid && p.has_res) ? p.res.at<bf16>(n, y, x, n0) : nullptr;
                tb_a[mt] = (valid && p.tbias) ? p.tbias + (size_t)n * p.tbias_pitch + n0 : nullptr;
                const bf16* pf = rrow_a[mt] ? rrow_a[mt] : ((p.accum && valid) ? orow_a[mt] : nullptr);
                if (pf) {
                    for (int c = blk_lo << 4; c < (blk_hi << 4); c += 64)
                        asm volatile("prefetch.global.L2 [%0];" ::"l"(pf + c));
                }
            }
            mbar_wait(&tfull[buf], bph);
            tc_fence_after();
            const uint32_t dbase = tmem_base + buf * (uint32_t)cols_per_buf;
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
                bf16* orow = orow_a[mt]; const bf16* rrow = rrow_a[mt]; const float* tb = tb_a[mt];
                const bool valid = orow != nullptr;
                // (staging the tile in shared memory to emit full 128-byte lines per store instruction was measured
                // SLOWER -- 153 vs 117 us at 96->96@64: the kernel is bound by L2 traffic, not store coalescing)
                // 64 output channels per trip: all TMEM / residual / accumulate loads of the trip are in flight
                // before the first use, so one L2 round trip is exposed per trip instead of per 16 columns
#pragma unroll 1
                constexpr int EB = 2;                         // 16-column blocks per trip (register budget: 320 threads)
                for (int blk = blk_lo; blk < blk_hi; blk += EB) {
                    uint32_t r[EB][16];
                    uint4 rr[EB][2], ra[EB][2];
#pragma unroll
                    for (int q = 0; q < EB; ++q) {
                        const int c = (blk + q) << 4;
                        if (blk + q < blk_hi) {
                            tmem_ld16(dbase + ((uint32_t)(qd * 32) << 16) + (uint32_t)(mt * p.NT + c), r[q]);
                            if (rrow) {
                                if (p.v256) { U8 t; ldg256(rrow + c, t); rr[q][0] = t.lo; rr[q][1] = t.hi; }
                                else { rr[q][0] = *reinterpret_cast<const uint4*>(rrow + c); rr[q][1] = *reinterpret_cast<const uint4*>(rrow + c + 8); }
                            }
                            if (p.accum && valid) {
                                if (p.v256) { U8 t; ldg256(orow + c, t); ra[q][0] = t.lo; ra[q][1] = t.hi; }
                                else { ra[q][0] = *reinterpret_cast<const uint4*>(orow + c); ra[q][1] = *reinterpret_cast<const uint4*>(orow + c + 8); }
                            }
                        }
                    }
                    tmem_ld_wait();
#pragma unroll
                    for (int q = 0; q < EB; ++q) {
                        const int c = (blk + q) << 4;
                        if (blk + q < blk_hi && valid && n0 + c < p.Cout) {
                            float v[16];
#pragma unroll
                            for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[q][i]);
                            if (p.bias) {
#pragma unroll
                                for (int i = 0; i < 16; i += 4) {                 // broadcast LDS.128 (all lanes, same address)
                                    const float4 b4 = *reinterpret_cast<const float4*>(sbias + n0 + c + i);
                                    v[i] += b4.x; v[i + 1] += b4.y; v[i + 2] += b4.z; v[i + 3] += b4.w;
                                }
                            }
                            if (tb) {
                                if (p.vec_tbias) {
#pragma unroll
                                    for (int i = 0; i < 16; i += 4) {
                                        const float4 b4 = __ldg(reinterpret_cast<const float4*>(tb + c + i));
                                        v[i] += b4.x; v[i + 1] += b4.y; v[i + 2] += b4.z; v[i + 3] += b4.w;
                                    }
                                } else {
#pragma unroll
                                    for (int i = 0; i < 16; ++i) v[i] += __ldg(tb + c + i);
                                }
                            }
                            if (rrow) {
                                const __nv_bfloat162* ha = reinterpret_cast<const __nv_bfloat162*>(&rr[q][0]);
                                const __nv_bfloat162* hb = reinterpret_cast<const __nv_bfloat162*>(&rr[q][1]);
#pragma unroll
                                for (int i = 0; i < 4; ++i) {
                                    float2 fa = __bfloat1622float2(ha[i]), fb = __bfloat1622float2(hb[i]);
                                    v[2 * i] += fa.x; v[2 * i + 1] += fa.y; v[8 + 2 * i] += fb.x; v[8 + 2 * i + 1] += fb.y;
                                }
                            }
                            if (p.accum) {
                                const __nv_bfloat162* ha = reinterpret_cast<const __nv_bfloat162*>(&ra[q][0]);
                                const __nv_bfloat162* hb = reinterpret_cast<const __nv_bfloat162*>(&ra[q][1]);
#pragma unroll
                                for (int i = 0; i < 4; ++i) {
                                    float2 fa = __bfloat1622float2(ha[i]), fb = __bfloat1622float2(hb[i]);
                                    v[2 * i] += fa.x; v[2 * i + 1] += fa.y; v[8 + 2 * i] += fb.x; v[8 + 2 * i + 1] += fb.y;
                                }
                            }
                            uint4 o0, o1;
                            __nv_bfloat162* h0 = reinterpret_cast<__nv_bfloat162*>(&o0);
                            __nv_bfloat162* h1 = reinterpret_cast<__nv_bfloat162*>(&o1);
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                h0[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
                                h1[i] = __floats2bfloat162_rn(v[8 + 2 * i], v[8 + 2 * i + 1]);
                            }
                            if (p.v256) stg256(orow + c, o0, o1);
                            else { *reinterpret_cast<uint4*>(orow + c) = o0; *reinterpret_cast<uint4*>(orow + c + 8) = o1; }
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(buf ? tempty_leader1 : tempty_leader0);
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                  // nobody exits (or frees TMEM) while the pair is still working
    if (warp == 1) { tc_fence_after(); tmem_dealloc2(tmem_base, 512u); }
}

int conv_tc_launch(const ddpm_conv_args* a, cudaStream_t st) {
    int rc = get_encode(); if (rc) return rc;
    Tc2Params p;
    p.out = TV(a->out);
    p.has_res = a->res.ptr != nullptr; p.res = p.has_res ? TV(a->res) : TV(a->out);
    p.bias = a->bias; p.tbias = a->tbias; p.tbias_pitch = a->tbias_pitch;
    p.bias_n = a->bias_n > 0 ? a->bias_n : a->out.C;
    p.Cin = a->in.C; p.Cout = a->out.C; p.NT = pick_nt(p.Cout);
    // Channel tiles of at most 128: with MT = 2 the weight slab is then shared by 256 pixel rows per CTA and the
    // A-patch halo is amortised over two M-tiles -> 26 % less L2->SM traffic per FLOP than NT = 192, MT = 1
    // (measured +8..14 % on every Cout = 192 layer); ddpm_set_tc_mode flag 32 keeps the wide tile.
    if (!(g_tc_exp & 32) && p.NT % 32 == 0 && p.NT > 128) p.NT /= 2;
    p.n_tiles = p.Cout / p.NT;
    p.taps = a->KH * a->KW;
    p.up = a->mode == DDPM_CONV_UP2X_PHASE ? 1 : 0; p.py = p.up ? (a->up_phase >> 1) : 0; p.px = p.up ? (a->up_phase & 1) : 0;
    p.Hp = a->in.H + 2; p.Wp = a->in.W + 2; p.H = a->in.H; p.W = a->in.W;
    p.Qtot = a->in.N * p.Hp * p.Wp;
    p.accum = (a->epi & DDPM_EPI_ACCUM) ? 1 : 0;
    p.sub = a->stride == 2 ? 1 : 0;
    p.vec_bias = a->bias && (((uintptr_t)a->bias & 15) == 0);
    p.vec_tbias = a->tbias && (((uintptr_t)a->tbias & 15) == 0) && (a->tbias_pitch % 4 == 0);
    p.v256 = (((uintptr_t)a->out.ptr & 31) == 0) && (a->out.pitch % 16 == 0) &&
             (!a->res.ptr || ((((uintptr_t)a->res.ptr & 31) == 0) && (a->res.pitch % 16 == 0))) && !(g_tc_exp & 128);
    int MT = 256 / p.NT; if (MT > 2) MT = 2; if (MT < 1) MT = 1;
    // small problems: prefer more, smaller items so that every SM pair gets one
    if (MT == 2 && (int64_t)ceil_div(p.Qtot, 512) * p.n_tiles < sm_count() / 2) MT = 1;
    const int halo_rows = p.taps > 1 ? p.Wp + 1 : 0;
    {
        int need = 128 * MT + 2 * halo_rows;
        int nseg = (need + 255) / 256;
        p.seg = (((need + nseg - 1) / nseg) + 7) & ~7;
        p.P = p.seg * nseg;
    }
    p.a_chunk_bytes = (p.P * 32 + 255) & ~255;
    p.b_chunk_bytes = p.taps * (p.NT / 2) * 32;             // multiple of 256: NT/2 is a multiple of 8
    const int KCH = p.Cin / KC;
    p.KS = p.taps > 1 ? 1 : (KCH < 4 ? KCH : 4);
    p.KCH2 = a->in2.ptr ? a->in2.C / KC : 0;                // fused 1x1 second operand (3x3 main conv only: KS == 1)
    p.b2_chunk_bytes = (p.NT / 2) * 32;
    const int budget = 212 * 1024;
    p.pix_tiles = ceil_div(p.Qtot, 256 * MT);
    p.items = p.pix_tiles * p.n_tiles;
    int pairs = sm_count() / 2; if (pairs > p.items) pairs = p.items; if (pairs < 1) pairs = 1;
    // Weights resident in shared memory when this CTA's half tile (all K-chunks, all taps) leaves room for a >= 3-deep
    // A ring and every CTA pair sees several items: then only activations stream (14.8 instead of 30.8 B/clk/SM at NT=96).
    p.b_res = 0;
    if (p.taps > 1 && !(g_tc_exp & 64)) {
        const int bres_bytes = KCH * p.b_chunk_bytes + p.KCH2 * p.b2_chunk_bytes;
        const int pr = pairs - pairs % p.n_tiles;             // a pair keeps ONE channel tile: pairs must be a multiple of n_tiles
        if (bres_bytes + 3 * p.a_chunk_bytes <= budget && pr >= p.n_tiles && p.items >= 3 * pr) { p.b_res = 1; pairs = pr; }
    }
    if (p.b_res) {
        p.stage_bytes = p.a_chunk_bytes;
        p.S = (budget - KCH * p.b_chunk_bytes - p.KCH2 * p.b2_chunk_bytes) / p.stage_bytes; if (p.S > 12) p.S = 12;
    } else {
        p.stage_bytes = (p.KS * (p.a_chunk_bytes + p.b_chunk_bytes) + 1023) & ~1023;
        p.S = budget / p.stage_bytes; if (p.S > 12) p.S = 12;
    }
    if (p.S < 2) return DDPM_E_ARG;
    size_t smem = (size_t)p.S * p.stage_bytes + (p.b_res ? (size_t)KCH * p.b_chunk_bytes + (size_t)p.KCH2 * p.b2_chunk_bytes : 0) +
                  8 * (2 * p.S + 4) + 16 + (size_t)p.Cout * 4 + 1024 + 16;

    CUtensorMap tmA, tmB, tmA2, tmB2;
    if (p.KCH2) {
        uint64_t da[2] = {(uint64_t)a->in2.C, (uint64_t)p.Qtot}; uint64_t sa[1] = {(uint64_t)a->in2.pitch * 2};
        uint32_t ba[2] = {KC, (uint32_t)p.seg};
        if (encode(&tmA2, a->in2.ptr, 2, da, sa, ba, CU_TENSOR_MAP_SWIZZLE_32B)) return 1;
        // 1x1 weights [Cout][1][Cin2] viewed as (c, n, tap = 1)
        uint64_t db[3] = {(uint64_t)a->in2.C, (uint64_t)p.Cout, 1};
        uint64_t sb[2] = {(uint64_t)a->in2.C * 2, (uint64_t)p.Cout * a->in2.C * 2};
        uint32_t bb[3] = {KC, (uint32_t)(p.NT / 2), 1};
        if (encode(&tmB2, (void*)a->w2, 3, db, sb, bb, CU_TENSOR_MAP_SWIZZLE_32B)) return 1;
    }
    {
        uint64_t da[2] = {(uint64_t)p.Cin, (uint64_t)p.Qtot}; uint64_t sa[1] = {(uint64_t)a->in.pitch * 2};
        uint32_t ba[2] = {KC, (uint32_t)p.seg};
        if (encode(&tmA, a->in.ptr, 2, da, sa, ba, CU_TENSOR_MAP_SWIZZLE_32B)) return 1;
        // weights [Cout][taps][Cin] viewed as (c, n, tap): one box brings all taps of NT/2 rows -> smem [tap][n][16 ch]
        uint64_t db[3] = {(uint64_t)p.Cin, (uint64_t)p.Cout, (uint64_t)p.taps};
        uint64_t sb[2] = {(uint64_t)p.taps * p.Cin * 2, (uint64_t)p.Cin * 2};
        uint32_t bb[3] = {KC, (uint32_t)(p.NT / 2), (uint32_t)p.taps};
        if (encode(&tmB, (void*)a->w, 3, db, sb, bb, CU_TENSOR_MAP_SWIZZLE_32B)) return 1;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * pairs); cfg.blockDim = dim3(TC2_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    static size_t configured[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#define TC2_GO(MTV, TAPSV, F2, SLOT) { \
        if (smem > configured[SLOT]) { CUDA_TRY(cudaFuncSetAttribute(conv_tc2_kernel<MTV, TAPSV, F2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); configured[SLOT] = smem; } \
        CUDA_TRY(cudaLaunchKernelEx(&cfg, conv_tc2_kernel<MTV, TAPSV, F2>, tmA, tmB, F2 ? tmA2 : tmA, F2 ? tmB2 : tmB, p)); }
    if (p.KCH2) { if (MT == 2) TC2_GO(2, 9, true, 4) else TC2_GO(1, 9, true, 5) }
    else if (p.taps == 4) { if (MT == 2) TC2_GO(2, 4, false, 6) else TC2_GO(1, 4, false, 7) }
    else if (MT == 2) { if (p.taps == 9) TC2_GO(2, 9, false, 0) else TC2_GO(2, 1, false, 1) }
    else { if (p.taps == 9) TC2_GO(1, 9, false, 2) else TC2_GO(1, 1, false, 3) }
#undef TC2_GO
    LAUNCH_OK();
    return 0;
}

// ================================================================================================
// weight gradient:  dW[co][ci][ky][kx] += sum_Q dY[Q][co] * A[Q + (ky-1)*Wp + (kx-1)][ci]
//
// The reduction runs over padded-linear pixels Q (dY's halo is zero, so halo rows contribute 0), which
// makes BOTH operands "MN-major" (channels contiguous, K = pixels strided): dY tiles [64 px][128 co]
// and activation patches [64+2 px][NT ci] are TMA-loaded with SWIZZLE_128B and fed to tcgen05.mma with
// a_major = b_major = MN.  A CTA owns one filter row ky (three taps = three row-shifted descriptors of
// the same patch, accumulators D[128 co][3*NT] in TMEM), one ci tile, one co tile and one slice of the
// pixel range (split-K).  Partials go to a workspace with coalesced stores and a second kernel reduces
// them into the fp32 OIHW gradient (no atomics).
// ================================================================================================
int wgrad_tc_supported(const ddpm_wgrad_args* a);
#define WG_KQ 64          // pixels per pipeline stage (4 UMMA K-steps)
#define WG_ROWS 72        // patch rows per stage (KQ + 2 shifts, rounded to 8)
#ifndef WG_STAGES
#define WG_STAGES 5
#endif

struct WgTcParams {
    float* ws;                  // [split][mtile][grp][128][3*NT]
    int Cin, Cout, NT, n_tiles, m_tiles;
    int Wp, Qtot, stages_total, stages_per_cta;
    int nblkA;                  // 64-channel blocks per activation patch (1 or 2)
    int stage_bytes, tmem_cols;
    int ntap;                   // taps per CTA: 3 (one filter row of a 3x3) or 1 (1x1)
    int CinV, CoutV;            // unpadded channel counts of the fp32 gradient
    // bias gradient for free: CTAs of group 0 run one extra N=16 MMA per K-step against a tile of ones,
    // D_bias[co][*] = sum_Q dY[Q][co] (halo rows of dY are zero), instead of a separate pass over dY
    float* ws_bias;             // [split][mtile][128] partials (NULL: no bias gradient)
    float* dbias;               // fp32 [CoutV], accumulated by the reduce kernel
};

__global__ void __launch_bounds__(TC_THREADS) wgrad_tc_kernel(const __grid_constant__ CUtensorMap tmY,
                                                               const __grid_constant__ CUtensorMap tmA, WgTcParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* ones = smem + (size_t)WG_STAGES * p.stage_bytes;            // [16 px][64 ch] of bf16 1.0 (2 KB, 1024-aligned)
    uint64_t* full = (uint64_t*)(ones + 2048);
    uint64_t* empty = full + WG_STAGES;
    uint64_t* acc_full = empty + WG_STAGES;
    uint32_t* tmem_slot = (uint32_t*)(acc_full + 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int split = blockIdx.x, mtile = blockIdx.z;
    const int ky = (int)blockIdx.y / p.n_tiles;
    const int ntile = (int)blockIdx.y - ky * p.n_tiles;
    const int grp = ky * p.n_tiles + ntile;                     // workspace / bias-dealing index
    // the K-steps of the bias reduction are dealt round-robin to the gridDim.y groups that stream the same dY
    // rows (putting all of them on group 0 made those CTAs the critical path: +11..16 % kernel time)
    const bool do_bias = p.ws_bias != nullptr;
    const int ngrp = gridDim.y;
    const int m0 = mtile * 128, n0 = ntile * p.NT;
    const int s_beg = split * p.stages_per_cta;
    const int s_end = min(p.stages_total, s_beg + p.stages_per_cta);
    const int nst = max(0, s_end - s_beg);
    const int y_bytes = 2 * WG_KQ * 128;                 // two 64-channel blocks of dY

    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmY) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
        for (int i = 0; i < WG_STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        mbar_init(acc_full, 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
    if (do_bias && warp >= 2) {
        for (int i = threadIdx.x - 64; i < 2048 / 4; i += TC_THREADS - 64) reinterpret_cast<uint32_t*>(ones)[i] = 0x3F803F80u;
        fence_proxy_async();                             // generic-proxy writes -> visible to the tensor core's async proxy
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t bias_col = (uint32_t)(p.ntap * p.NT);

    if (warp == 0) {
        if (lane == 0) {
            for (int i = 0; i < nst; ++i) {
                const int s = i % WG_STAGES; const uint32_t ph = (i / WG_STAGES) & 1;
                mbar_wait(&empty[s], ph ^ 1);
                uint8_t* dst = smem + (size_t)s * p.stage_bytes;
                mbar_expect_tx(&full[s], (uint32_t)(y_bytes + p.nblkA * WG_ROWS * 128));
                const int Q = (s_beg + i) * WG_KQ;
                tma_load_2d(dst, &tmY, &full[s], m0, Q);
                tma_load_2d(dst + WG_KQ * 128, &tmY, &full[s], m0 + 64, Q);
                const int rowA = p.ntap == 3 ? Q + (ky - 1) * p.Wp - 1 : Q;
                for (int b = 0; b < p.nblkA; ++b)
                    tma_load_2d(dst + y_bytes + (size_t)b * WG_ROWS * 128, &tmA, &full[s], n0 + 64 * b, rowA);
            }
        }
    } else if (warp == 1) {
        {   // whole warp, warp-uniform control flow; one elected lane issues tcgen05 instructions
            const bool el = elect_one();
            // a_major = b_major = MN (bits 15, 16); M = 128; N = NT
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) |
                                   ((uint32_t)(p.NT >> 3) << 17) | ((128u >> 4) << 24);
            const uint32_t hi = desc_hi(1024u, 2u);                      // SBO 1024 B, SWIZZLE_128B
            const uint32_t y_lo0 = desc_lo(smem_u32(smem), (uint32_t)(WG_KQ * 128));
            const uint32_t a_lo0 = desc_lo(smem_u32(smem) + (uint32_t)y_bytes, (uint32_t)(WG_ROWS * 128));
            const uint32_t stage16 = (uint32_t)(p.stage_bytes >> 4);
            const bool three = p.ntap == 3;
            const uint32_t idesc_b = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((16u >> 3) << 17) | ((128u >> 4) << 24);
            const uint64_t ones_desc = desc_pack(desc_lo(smem_u32(ones), 2048u), hi);
            // two copies of the loop: a predicated-off bias MMA in the common loop cost 11 % (measured A/B)
            auto run = [&](auto with_bias, auto with_three) {
                constexpr bool BIAS = decltype(with_bias)::value, THREE = decltype(with_three)::value;
                uint32_t acc = 0, accb = 0;
                int kmod = ((s_beg * (WG_KQ / 16)) % ngrp);                 // (global K-step index) mod ngrp
                for (int i = 0; i < nst; ++i) {
                    const uint32_t s = (uint32_t)(i % WG_STAGES); const uint32_t ph = (i / WG_STAGES) & 1;
                    mbar_wait(&full[s], ph);
                    tc_fence_after();
                    const uint32_t y_lo = y_lo0 + s * stage16, a_lo = a_lo0 + s * stage16;
#pragma unroll
                    for (int ks = 0; ks < WG_KQ / 16; ++ks) {
                        const uint64_t ydesc = desc_pack(y_lo + (uint32_t)(ks * 16 * 128 / 16), hi);
                        if (el) umma_bf16(tmem_base, ydesc, desc_pack(a_lo + (uint32_t)((ks * 16) * 8), hi), idesc, ks == 0 ? acc : 1u);
                        if (THREE && el) {
                            umma_bf16(tmem_base + (uint32_t)p.NT, ydesc, desc_pack(a_lo + (uint32_t)((ks * 16 + 1) * 8), hi), idesc, ks == 0 ? acc : 1u);
                            umma_bf16(tmem_base + (uint32_t)(2 * p.NT), ydesc, desc_pack(a_lo + (uint32_t)((ks * 16 + 2) * 8), hi), idesc, ks == 0 ? acc : 1u);
                        }
                        if (BIAS) {
                            if (kmod == grp) { if (el) umma_bf16(tmem_base + bias_col, ydesc, ones_desc, idesc_b, accb); accb = 1; }
                            if (++kmod == ngrp) kmod = 0;
                        }
                    }
                    acc = 1;
                    if (el) umma_commit(&empty[s]);
                    __syncwarp();
                }
            };
            // every run-time flag of the issue loop is a compile-time constant of its copy (the loop is that sensitive)
            if (do_bias) { if (three) run(std::true_type{}, std::true_type{}); else run(std::true_type{}, std::false_type{}); }
            else { if (three) run(std::false_type{}, std::true_type{}); else run(std::false_type{}, std::false_type{}); }
            if (el) umma_commit(acc_full);
            __syncwarp();
        }
    } else {
        const int qd = warp & 3;
        mbar_wait(acc_full, 0);
        tc_fence_after();
        const int cols = p.ntap * p.NT;
        float* dst = p.ws + ((((size_t)split * p.m_tiles + mtile) * gridDim.y + grp) * 128 + qd * 32 + lane) * cols;
#pragma unroll 1
        for (int c0 = 0; c0 < cols; c0 += 16) {
            uint32_t r[16];
            if (nst > 0) {
                tmem_ld16(tmem_base + ((uint32_t)(qd * 32) << 16) + (uint32_t)c0, r);
                tmem_ld_wait();
            } else {
#pragma unroll
                for (int i = 0; i < 16; ++i) r[i] = 0u;
            }
#pragma unroll
            for (int i = 0; i < 16; i += 4)
                *reinterpret_cast<uint4*>(dst + c0 + i) = make_uint4(r[i], r[i + 1], r[i + 2], r[i + 3]);
        }
        if (do_bias) {
            uint32_t r[16];
            // this CTA ran a bias MMA iff one of its K-steps k in [s_beg*4, s_end*4) has k % ngrp == grp
            const int k0 = s_beg * (WG_KQ / 16), k1 = s_end * (WG_KQ / 16);
            const int first = k0 + ((grp - k0 % ngrp) % ngrp + ngrp) % ngrp;
            if (nst > 0 && first < k1) { tmem_ld16(tmem_base + ((uint32_t)(qd * 32) << 16) + bias_col, r); tmem_ld_wait(); }
            else r[0] = 0u;
            p.ws_bias[(((size_t)split * ngrp + grp) * p.m_tiles + mtile) * 128 + qd * 32 + lane] = __uint_as_float(r[0]);
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 1) { tc_fence_after(); tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols); }
}

// ================================================================================================
// Pair variant of the weight gradient (cta_group::2): the two output-channel tiles of a layer with Cout in (128, 256]
// (or each pair of tiles for wider layers) are computed by the two CTAs of a cluster as ONE M = 256 MMA.
//
// Why (ncu, profiles/r2_ncu_prof_wgrad_192_32.txt): the single-CTA kernel receives 966 MB through the L2->SM crossbar
// for 114 MB of tensors at 192->192@32 -- 39 B/clk per SM, 92 % of the ~42 B/clk/SM the fabric sustains -- with the
// tensor pipe 65 % active and the shared-memory banks only 38 % (reads) + 16 % (writes) busy: it is bound by operand
// INGEST per SM, not by shared-memory bandwidth (round 1's reading).  Per 64-pixel stage a CTA took in 16 KB of dY and
// 18.4 KB of activation patch.  Here each CTA still stages its own dY tile (its 128 output channels = its half of M)
// but only HALF of the patch channels (N/2); both tensor cores read both halves -> 25.2 KB per stage and CTA (-27 %),
// and one more pipeline stage fits.  Barrier protocol as in conv_tc2_kernel: full[s] lives in the leader and collects
// the bytes of both CTAs, empty[s] / acc_full are tcgen05.commit multicasts to both.
// The epilogue, the workspace layout and the reduce kernel are those of the single-CTA kernel.
// ================================================================================================
#define WG2_STAGES 6
__global__ void __launch_bounds__(TC_THREADS) wgrad_tc2_kernel(const __grid_constant__ CUtensorMap tmY,
                                                                const __grid_constant__ CUtensorMap tmA, WgTcParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* ones = smem + (size_t)WG2_STAGES * p.stage_bytes;           // [16 px][64 ch] of bf16 1.0 (2 KB, 1024-aligned)
    uint64_t* full = (uint64_t*)(ones + 2048);
    uint64_t* empty = full + WG2_STAGES;
    uint64_t* acc_full = empty + WG2_STAGES;
    uint32_t* tmem_slot = (uint32_t*)(acc_full + 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();                    // cluster (2,1,1): rank = blockIdx.x & 1 = which tile of the pair
    const bool leader = rank == 0;
    const int split = blockIdx.z, mtile = blockIdx.x;            // (grid = m_tiles x groups x splits: the pair sits on x like conv_tc2's)
    const int ky = (int)blockIdx.y / p.n_tiles;
    const int ntile = (int)blockIdx.y - ky * p.n_tiles;
    const int grp = ky * p.n_tiles + ntile;
    const bool do_bias = p.ws_bias != nullptr;
    const int ngrp = gridDim.y;
    const int m0 = mtile * 128, n0 = ntile * p.NT + (int)rank * (p.NT / 2);
    const int s_beg = split * p.stages_per_cta;
    const int s_end = min(p.stages_total, s_beg + p.stages_per_cta);
    const int nst = max(0, s_end - s_beg);
    const int y_bytes = 2 * WG_KQ * 128;                 // two 64-channel blocks of dY

    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmY) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
        for (int i = 0; i < WG2_STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        mbar_init(acc_full, 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc2(tmem_slot, (uint32_t)p.tmem_cols);
    if (do_bias && warp >= 2) {
        for (int i = threadIdx.x - 64; i < 2048 / 4; i += TC_THREADS - 64) reinterpret_cast<uint32_t*>(ones)[i] = 0x3F803F80u;
        fence_proxy_async();
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                  // the peer's barriers are initialised before anyone signals them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t bias_col = (uint32_t)(p.ntap * p.NT);

    if (warp == 0) {
        // ===================================================================== TMA producer (both CTAs)
        if (lane == 0) {
            for (int i = 0; i < nst; ++i) {
                const int s = i % WG2_STAGES; const uint32_t ph = (i / WG2_STAGES) & 1;
                mbar_wait(&empty[s], ph ^ 1);
                uint8_t* dst = smem + (size_t)s * p.stage_bytes;
                const uint32_t fbar = mapa_u32(smem_u32(&full[s]), 0);
                if (leader) mbar_expect_tx(&full[s], (uint32_t)(2 * (y_bytes + WG_ROWS * 128)));
                const int Q = (s_beg + i) * WG_KQ;
                tma2_load_2d(dst, &tmY, fbar, m0, Q);
                tma2_load_2d(dst + WG_KQ * 128, &tmY, fbar, m0 + 64, Q);
                const int rowA = p.ntap == 3 ? Q + (ky - 1) * p.Wp - 1 : Q;
                tma2_load_2d(dst + y_bytes, &tmA, fbar, n0, rowA);
            }
        }
    } else if (warp == 1) {
        // ===================================================================== MMA issuer (leader CTA only)
        if (leader) {
            const bool el = elect_one();
            // a_major = b_major = MN (bits 15, 16); M = 256 over the pair; N = NT (each CTA holds NT/2 patch channels)
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) |
                                   ((uint32_t)(p.NT >> 3) << 17) | ((256u >> 4) << 24);
            const uint32_t hi = desc_hi(1024u, 2u);                      // SBO 1024 B, SWIZZLE_128B
            const uint32_t y_lo0 = desc_lo(smem_u32(smem), (uint32_t)(WG_KQ * 128));
            const uint32_t a_lo0 = desc_lo(smem_u32(smem) + (uint32_t)y_bytes, (uint32_t)(WG_ROWS * 128));
            const uint32_t stage16 = (uint32_t)(p.stage_bytes >> 4);
            const bool three = p.ntap == 3;
            const uint32_t idesc_b = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((16u >> 3) << 17) | ((256u >> 4) << 24);
            const uint64_t ones_desc = desc_pack(desc_lo(smem_u32(ones), 2048u), hi);
            auto run = [&](auto with_bias, auto with_three) {
                constexpr bool BIAS = decltype(with_bias)::value, THREE = decltype(with_three)::value;
                uint32_t acc = 0, accb = 0;
                int kmod = ((s_beg * (WG_KQ / 16)) % ngrp);
                for (int i = 0; i < nst; ++i) {
                    const uint32_t s = (uint32_t)(i % WG2_STAGES); const uint32_t ph = (i / WG2_STAGES) & 1;
                    mbar_wait(&full[s], ph);
                    tc_fence_after();
                    const uint32_t y_lo = y_lo0 + s * stage16, a_lo = a_lo0 + s * stage16;
#pragma unroll
                    for (int ks = 0; ks < WG_KQ / 16; ++ks) {
                        const uint64_t ydesc = desc_pack(y_lo + (uint32_t)(ks * 16 * 128 / 16), hi);
                        if (el) umma2_bf16(tmem_base, ydesc, desc_pack(a_lo + (uint32_t)((ks * 16) * 8), hi), idesc, ks == 0 ? acc : 1u);
                        if (THREE && el) {
                            umma2_bf16(tmem_base + (uint32_t)p.NT, ydesc, desc_pack(a_lo + (uint32_t)((ks * 16 + 1) * 8), hi), idesc, ks == 0 ? acc : 1u);
                            umma2_bf16(tmem_base + (uint32_t)(2 * p.NT), ydesc, desc_pack(a_lo + (uint32_t)((ks * 16 + 2) * 8), hi), idesc, ks == 0 ? acc : 1u);
                        }
                        if (BIAS) {
                            if (kmod == grp) { if (el) umma2_bf16(tmem_base + bias_col, ydesc, ones_desc, idesc_b, accb); accb = 1; }
                            if (++kmod == ngrp) kmod = 0;
                        }
                    }
                    acc = 1;
                    if (el) umma2_commit_mc(&empty[s]);
                    __syncwarp();
                }
            };
            if (do_bias) { if (three) run(std::true_type{}, std::true_type{}); else run(std::true_type{}, std::false_type{}); }
            else { if (three) run(std::false_type{}, std::true_type{}); else run(std::false_type{}, std::false_type{}); }
            if (el) umma2_commit_mc(acc_full);
            __syncwarp();
        }
    } else {
        // ===================================================================== epilogue (both CTAs: own 128 output channels)
        const int qd = warp & 3;
        mbar_wait(acc_full, 0);
        tc_fence_after();
        const int cols = p.ntap * p.NT;
        float* dst = p.ws + ((((size_t)split * p.m_tiles + mtile) * gridDim.y + grp) * 128 + qd * 32 + lane) * cols;
#pragma unroll 1
        for (int c0 = 0; c0 < cols; c0 += 16) {
            uint32_t r[16];
            if (nst > 0) {
                tmem_ld16(tmem_base + ((uint32_t)(qd * 32) << 16) + (uint32_t)c0, r);
                tmem_ld_wait();
            } else {
#pragma unroll
                for (int i = 0; i < 16; ++i) r[i] = 0u;
            }
#pragma unroll
            for (int i = 0; i < 16; i += 4)
                *reinterpret_cast<uint4*>(dst + c0 + i) = make_uint4(r[i], r[i + 1], r[i + 2], r[i + 3]);
        }
        if (do_bias) {
            uint32_t r[16];
            const int k0 = s_beg * (WG_KQ / 16), k1 = s_end * (WG_KQ / 16);
            const int first = k0 + ((grp - k0 % ngrp) % ngrp + ngrp) % ngrp;
            if (nst > 0 && first < k1) { tmem_ld16(tmem_base + ((uint32_t)(qd * 32) << 16) + bias_col, r); tmem_ld_wait(); }
            else r[0] = 0u;
            p.ws_bias[(((size_t)split * ngrp + grp) * p.m_tiles + mtile) * 128 + qd * 32 + lane] = __uint_as_float(r[0]);
        }
        tc_fence_before();
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                  // nobody exits (or frees TMEM) while the pair is still working
    if (warp == 1) { tc_fence_after(); tmem_dealloc2(tmem_base, (uint32_t)p.tmem_cols); }
}

// dw[co][ci][ky][kx] += sum_split ws[split][mtile][ky*n_tiles+ntile][co%128][kx*NT + ci%NT]
__global__ void wgrad_reduce_kernel(const float* __restrict__ ws, float* __restrict__ dw, int splits, WgTcParams p) {
    const int gtid = blockIdx.x * blockDim.x + threadIdx.x, gthreads = gridDim.x * blockDim.x;
    const int taps = p.ntap * p.ntap;
    const int total = p.CoutV * taps * p.CinV;
    const int grps = p.ntap * p.n_tiles, cols = p.ntap * p.NT;
    for (int i = gtid; i < total; i += gthreads) {
        // enumerate (co, tap, ci) with ci fastest so workspace reads are coalesced
        int ci = i % p.CinV; int r = i / p.CinV; int tap = r % taps; int co = r / taps;
        int ky = tap / p.ntap, kx = tap - ky * p.ntap;
        int mtile = co >> 7, ntile = ci / p.NT;
        size_t off = ((((size_t)mtile) * grps + ky * p.n_tiles + ntile) * 128 + (co & 127)) * cols + kx * p.NT + (ci - ntile * p.NT);
        size_t stride = (size_t)p.m_tiles * grps * 128 * cols;
        // four independent partial sums: the loads of a thread are independent instead of one dependent chain per
        // split (the kernel is latency-bound: ~80 k outputs x 12-49 splits); fixed order -> still deterministic
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
        const float* w0 = ws + off;
        int s = 0;
        for (; s + 4 <= splits; s += 4) {
            a0 += w0[(size_t)s * stride]; a1 += w0[(size_t)(s + 1) * stride];
            a2 += w0[(size_t)(s + 2) * stride]; a3 += w0[(size_t)(s + 3) * stride];
        }
        for (; s < splits; ++s) a0 += w0[(size_t)s * stride];
        dw[((size_t)co * p.CinV + ci) * taps + tap] += (a0 + a1) + (a2 + a3);
    }
    if (p.ws_bias && p.dbias) {                              // one warp per output channel, lanes stride over the partials
        const int lane = gtid & 31, nwarp = gthreads >> 5;
        for (int co = gtid >> 5; co < p.CoutV; co += nwarp) {
            float acc = 0.f;
            for (int s = lane; s < splits * grps; s += 32) acc += p.ws_bias[((size_t)s * p.m_tiles + (co >> 7)) * 128 + (co & 127)];
            acc = warp_sum(acc);
            if (lane == 0) p.dbias[co] += acc;
        }
    }
}

static int sm_count() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    }
    return n;
}

static int wg_pick_nt(int Cin) {
    for (int nt = 128; nt >= 16; nt -= 16) if (Cin % nt == 0) return nt;
    return 0;
}

static int wg_pair(const WgTcParams& p) {
    // the pair kernel: an even number of 128-row output-channel tiles (Cout in (128,256], (384,512], ...); ddpm_set_tc_mode
    // flag 1024 turns it off (A/B against the single-CTA kernel).
    if (g_tc_exp & 1024) return 0;
    // Measured (profiles/r2_kbench_wgrad_pair_vs_single.txt): -9 % on the large Cout = 192 layers, +5 % on 384->192 @ 16 / 8
    // (four ci tiles x few pixels: the halved split count costs more than the smaller patch saves) -> small problems with
    // many ci tiles stay on the single-CTA kernel.
    if (p.n_tiles > 2 && p.stages_total < 1500) return 0;
    return (p.m_tiles % 2 == 0) && p.NT % 16 == 0;
}
static void wg_plan(const ddpm_wgrad_args* a, WgTcParams* p, int* splits) {
    p->Cin = a->act.C; p->Cout = a->dy.C; p->NT = wg_pick_nt(p->Cin);
    p->ntap = a->KH == 3 ? 3 : 1;
    p->CinV = a->cin_valid > 0 ? a->cin_valid : p->Cin; p->CoutV = a->cout_valid > 0 ? a->cout_valid : p->Cout;
    p->n_tiles = p->Cin / p->NT; p->m_tiles = (p->Cout + 127) / 128;
    p->Wp = a->act.W + 2; p->Qtot = a->act.N * (a->act.H + 2) * p->Wp;
    p->stages_total = (p->Qtot + WG_KQ - 1) / WG_KQ;
    p->nblkA = (p->NT + 63) / 64;
    p->stage_bytes = 2 * WG_KQ * 128 + p->nblkA * WG_ROWS * 128;
    p->tmem_cols = 32; while (p->tmem_cols < p->ntap * p->NT + 16) p->tmem_cols <<= 1;
    int yz = p->ntap * p->n_tiles * p->m_tiles;
    // one CTA per SM (176 KB of shared memory): the grid must not exceed ONE wave, or the second,
    // nearly empty wave doubles the kernel's duration -> floor, not ceil
    int sp = sm_count() / yz;
    int max_sp = (p->stages_total + 7) / 8; if (max_sp < 1) max_sp = 1;
    if (sp > max_sp) sp = max_sp;
    if (sp < 1) sp = 1;
    p->stages_per_cta = (p->stages_total + sp - 1) / sp;
    *splits = (p->stages_total + p->stages_per_cta - 1) / p->stages_per_cta;
    if (wg_pair(*p)) p->stage_bytes = 2 * WG_KQ * 128 + WG_ROWS * 128;      // own dY tile + HALF of the patch channels (one 64-channel box)
}

extern "C" int64_t ddpm_wgrad_workspace_bytes(const ddpm_wgrad_args* a) {
    if (!a || !wgrad_tc_supported(a)) return 0;
    WgTcParams p; int splits; wg_plan(a, &p, &splits);
    return (int64_t)splits * p.m_tiles * p.ntap * p.n_tiles * 128 * p.ntap * p.NT * 4 + (int64_t)splits * p.ntap * p.n_tiles * p.m_tiles * 128 * 4;
}

int wgrad_tc_supported(const ddpm_wgrad_args* a) {
    if (a->dtype != DDPM_BF16 || a->stride != 1 || a->a_silu) return 0;
    if (!((a->KH == 3 && a->KW == 3 && a->pad == 1) || (a->KH == 1 && a->KW == 1 && a->pad == 0))) return 0;
    const ddpm_tensor &x = a->act, &y = a->dy;
    if (x.halo != 1 || y.halo != 1 || x.H != y.H || x.W != y.W || x.N != y.N) return 0;
    if (x.C % 16 || y.C % 8 || x.pitch % 8 || y.pitch % 8) return 0;
    if (((uintptr_t)x.ptr & 15) || ((uintptr_t)y.ptr & 15)) return 0;
    if (wg_pick_nt(x.C) == 0) return 0;
    if ((int64_t)x.N * (x.H + 2) * (x.W + 2) < 8 * WG_KQ) return 0;      // tiny problems: CUDA cores
    return 1;
}

int wgrad_tc_launch(const ddpm_wgrad_args* a, cudaStream_t st) {
    int rc = get_encode(); if (rc) return rc;
    WgTcParams p; int splits; wg_plan(a, &p, &splits);
    const int64_t main_bytes = (int64_t)splits * p.m_tiles * p.ntap * p.n_tiles * 128 * p.ntap * p.NT * 4;
    int64_t need = main_bytes + (int64_t)splits * p.ntap * p.n_tiles * p.m_tiles * 128 * 4;
    if (!a->workspace || a->workspace_bytes < need) return DDPM_E_ARG;
    p.ws = (float*)a->workspace;
    p.dbias = a->dbias;
    p.ws_bias = a->dbias ? (float*)((char*)a->workspace + main_bytes) : nullptr;
    CUtensorMap tmY, tmA;
    {
        uint64_t d[2] = {(uint64_t)p.Cout, (uint64_t)p.Qtot}; uint64_t s[1] = {(uint64_t)a->dy.pitch * 2};
        uint32_t b[2] = {64, WG_KQ};
        if (encode(&tmY, a->dy.ptr, 2, d, s, b, CU_TENSOR_MAP_SWIZZLE_128B)) return 1;
    }
    {
        uint64_t d[2] = {(uint64_t)p.Cin, (uint64_t)p.Qtot}; uint64_t s[1] = {(uint64_t)a->act.pitch * 2};
        uint32_t b[2] = {64, WG_ROWS};
        if (encode(&tmA, a->act.ptr, 2, d, s, b, CU_TENSOR_MAP_SWIZZLE_128B)) return 1;
    }
    if (wg_pair(p)) {
        const size_t smem2 = (size_t)WG2_STAGES * p.stage_bytes + 2048 + 8 * (2 * WG2_STAGES + 1) + 16 + 1024;
        static size_t configured2 = 0;
        if (smem2 > configured2) {
            CUDA_TRY(cudaFuncSetAttribute(wgrad_tc2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
            configured2 = smem2;
        }
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(p.m_tiles, p.ntap * p.n_tiles, splits); cfg.blockDim = dim3(TC_THREADS); cfg.dynamicSmemBytes = smem2; cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        CUDA_TRY(cudaLaunchKernelEx(&cfg, wgrad_tc2_kernel, tmY, tmA, p));
    } else {
        const size_t smem = (size_t)WG_STAGES * p.stage_bytes + 2048 + 8 * (2 * WG_STAGES + 1) + 16 + 1024;
        static size_t configured = 0;
        if (smem > configured) {
            CUDA_TRY(cudaFuncSetAttribute(wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            configured = smem;
        }
        CUDA_TRY(launch_kernel(wgrad_tc_kernel, dim3(splits, p.ntap * p.n_tiles, p.m_tiles), dim3(TC_THREADS), smem, st, tmY, tmA, p));
    }
    LAUNCH_OK();
    int total = p.CoutV * p.ntap * p.ntap * p.CinV;
    int rg = (total + 255) / 256; if (rg > 148 * 8) rg = 148 * 8;
    CUDA_TRY(launch_kernel(wgrad_reduce_kernel, dim3(rg), dim3(256), 0, st, (const float*)p.ws, a->dw, splits, p));
    LAUNCH_OK();
    return 0;
}
