// Shared device/host helpers for libddpm_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include "../../include/ddpm_b200.h"

typedef __nv_bfloat16 bf16;

extern int64_t g_ddpm_launches;  // counted by LAUNCH_OK (host side, single-threaded use)

#define LAUNCH_OK()                                   \
    do {                                              \
        ++g_ddpm_launches;                            \
        cudaError_t e__ = cudaGetLastError();         \
        if (e__ != cudaSuccess) return (int)e__;      \
    } while (0)

#define CUDA_TRY(x)                                   \
    do {                                              \
        cudaError_t e__ = (x);                        \
        if (e__ != cudaSuccess) return (int)e__;      \
    } while (0)

static inline int ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

template <typename... KA, typename... A>
static inline cudaError_t launch_kernel(void (*kernel)(KA...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, A&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KA>(args)...);
}

template <typename T> struct Cvt;
template <> struct Cvt<float> {
    __device__ __forceinline__ static float ld(const float* p) { return *p; }
    __device__ __forceinline__ static void st(float* p, float v) { *p = v; }
};
template <> struct Cvt<bf16> {
    __device__ __forceinline__ static float ld(const bf16* p) { return __bfloat162float(*p); }
    __device__ __forceinline__ static void st(bf16* p, float v) { *p = __float2bfloat16_rn(v); }
};
template <typename T> __device__ __forceinline__ float ldf(const T* p) { return Cvt<T>::ld(p); }
template <typename T> __device__ __forceinline__ void stf(T* p, float v) { Cvt<T>::st(p, v); }

// 8-element (bf16) / 4-element (fp32) 16-byte vectors of activations
template <typename T> struct Vec16;
template <> struct Vec16<float> {
    static constexpr int N = 4;
    float v[4];
    __device__ __forceinline__ void load(const float* p) {
        float4 t = *reinterpret_cast<const float4*>(p);
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    }
    __device__ __forceinline__ void store(float* p) const {
        *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    }
};
template <> struct Vec16<bf16> {
    static constexpr int N = 8;
    float v[8];
    __device__ __forceinline__ void load(const bf16* p) {
        uint4 t = *reinterpret_cast<const uint4*>(p);
        const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&t);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            float2 f = __bfloat1622float2(h[i]);
            v[2 * i] = f.x; v[2 * i + 1] = f.y;
        }
    }
    __device__ __forceinline__ void store(bf16* p) const {
        uint4 t;
        __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&t);
#pragma unroll
        for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
        *reinterpret_cast<uint4*>(p) = t;
    }
};

// SiLU via ex2.approx + rcp.approx: 2 MUFU + 3 FP32 instructions per element (~2 ulp, far inside the 1e-4
// fp32 parity budget).  __expf / __fdividef expand to range-checked sequences (FSETP/FSEL/extra FMULs) that
// doubled the instruction count of the GroupNorm kernels, which are issue-bound on B200.
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float sigmoid_f(float z) { return rcp_approx(1.0f + ex2_approx(-1.4426950408889634f * z)); }
__device__ __forceinline__ float silu_f(float z) { return z * sigmoid_f(z); }
__device__ __forceinline__ float dsilu_f(float z) {
    const float s = sigmoid_f(z);
    return fmaf(z * (1.0f - s), s, s);          // s * (1 + z (1 - s))
}

// bf16 activation paths: SiLU through ONE MUFU (tanh.approx, relative error 2^-11) instead of ex2 + rcp:
//   with h = z/2:  silu(z) = h + h*tanh(h);   silu'(z) = s + s*h*(1 - tanh(h)),  s = 0.5 + 0.5*tanh(h)
// 3 (forward) / 6 (derivative) instructions including the affine that produces h, against 6 / 9.  Absolute error
// <= |z| * 2.5e-4 -- below the bf16 resolution of the tensors these kernels write; the fp32 kernels keep silu_f.
__device__ __forceinline__ float tanh_approx(float x) { float y; asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float silu_half(float h) { return fmaf(h, tanh_approx(h), h); }
__device__ __forceinline__ float dsilu_half(float h) {
    const float t = tanh_approx(h);
    const float s = fmaf(0.5f, t, 0.5f);
    return fmaf(s, h * (1.0f - t), s);
}

// same with the 1/(1-p) of a following dropout folded into the constants: hs = 0.5 / (1 - p)
__device__ __forceinline__ float dsilu_half_scaled(float h, float hs) {
    const float t = tanh_approx(h);
    const float s = fmaf(hs, t, hs);
    return fmaf(s, h * (1.0f - t), s);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// NHWC view addressing (see ddpm_b200.h)
struct TV {
    char* ptr;
    int N, H, W, C, pitch, halo;
    int Hp, Wp;
    __host__ __device__ TV() {}
    __host__ __device__ explicit TV(const ddpm_tensor& t)
        : ptr((char*)t.ptr), N(t.N), H(t.H), W(t.W), C(t.C), pitch(t.pitch), halo(t.halo),
          Hp(t.H + 2 * t.halo), Wp(t.W + 2 * t.halo) {}
    __device__ __forceinline__ int64_t pix(int n, int y, int x) const {
        return ((int64_t)(n * Hp + y + halo) * Wp + x + halo) * pitch;
    }
    template <typename T> __device__ __forceinline__ T* at(int n, int y, int x, int c = 0) const {
        return reinterpret_cast<T*>(ptr) + pix(n, y, x) + c;
    }
};

static inline bool tensor_ok(const ddpm_tensor* t) {
    return t && t->ptr && t->N > 0 && t->H > 0 && t->W > 0 && t->C > 0 && t->pitch >= t->C &&
           (t->halo == 0 || t->halo == 1);
}

// Philox4x32-10 counter RNG (dropout masks; recomputed in backward from the same counters)
__device__ __forceinline__ uint4 philox4(uint32_t k0, uint32_t k1, uint4 c) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
        uint32_t hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
        c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
        k0 += W0; k1 += W1;
    }
    return c;
}
// keep-bits for VEC consecutive elements starting at `e0` (e0 % VEC == 0 for VEC in {4, 8}): one
// Philox call per 4 elements; bit i set = keep element e0+i.  Same function in forward and backward.
template <int VEC>
__device__ __forceinline__ uint32_t dropout_mask(const uint64_t* rng, uint32_t layer, uint64_t e0, float p) {
    const uint64_t seed = rng[0], step = rng[1];
    const uint32_t thr = (uint32_t)(p * 16777216.0f);            // keep iff (w >> 8) >= thr
    uint32_t m = 0;
    if (VEC == 1) {
        uint4 r = philox4((uint32_t)seed, (uint32_t)(seed >> 32),
                          make_uint4((uint32_t)(e0 >> 2), (uint32_t)(e0 >> 34), (uint32_t)step, layer));
        uint32_t w = (e0 & 3) == 0 ? r.x : (e0 & 3) == 1 ? r.y : (e0 & 3) == 2 ? r.z : r.w;
        return (w >> 8) >= thr ? 1u : 0u;
    }
#pragma unroll
    for (int q = 0; q < VEC / 4; ++q) {
        uint64_t e = (e0 >> 2) + q;
        uint4 r = philox4((uint32_t)seed, (uint32_t)(seed >> 32),
                          make_uint4((uint32_t)e, (uint32_t)(e >> 32), (uint32_t)step, layer));
        m |= ((r.x >> 8) >= thr ? 1u : 0u) << (4 * q);
        m |= ((r.y >> 8) >= thr ? 1u : 0u) << (4 * q + 1);
        m |= ((r.z >> 8) >= thr ? 1u : 0u) << (4 * q + 2);
        m |= ((r.w >> 8) >= thr ? 1u : 0u) << (4 * q + 3);
    }
    return m;
}
// Dropout keep-bits.  The GroupNorm kernels are instruction-bound on B200 (an SM has ~22 B/clk of HBM
// bandwidth, i.e. a budget of ~20 instructions per bf16 element), and Philox4x32-10 cost ~12 of them.
// Parity with ATen's mask is statistical only (SURVEY.md §7), so the mask comes from a counter hash:
// element e uses 16-bit half (e & 1) of lowbias32((e >> 1) ^ key), key = f(seed, step, layer); keep iff
// half >= thr16 = round(p * 65536).  ~4 instructions per element; fp32 (VEC 4), bf16 (VEC 8) and scalar paths
// draw the same mask; forward and backward recompute it from the same (seed, step, layer, index).
__device__ __forceinline__ uint32_t lowbias32(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
    return x;
}
__device__ __forceinline__ uint32_t dropout_key(const uint64_t* rng, uint32_t layer) {
    const uint64_t seed = rng[0], step = rng[1];
    uint32_t k = lowbias32((uint32_t)seed ^ 0x9E3779B9U);
    k = lowbias32(k ^ (uint32_t)(seed >> 32));
    k = lowbias32(k + (uint32_t)step * 0x85EBCA6BU);
    k = lowbias32(k ^ (layer * 0xC2B2AE35U));
    return k;
}
// in-place: v[i] = keep_i ? v[i] * scale : 0 for the VEC elements starting at (wrapping 32-bit) index e0
template <int VEC>
__device__ __forceinline__ void dropout_apply(float* v, uint32_t key, uint32_t e0, uint32_t thr16, float scale) {
    const uint32_t base = (e0 >> 1) ^ key;
    if (VEC == 1) {
        const uint32_t h = lowbias32(base);
        v[0] = (((e0 & 1) ? (h >> 16) : (h & 0xffffu)) >= thr16) ? v[0] * scale : 0.f;
        return;
    }
#pragma unroll
    for (int i = 0; i < VEC / 2; ++i) {
        const uint32_t h = lowbias32(base + (uint32_t)i);
        v[2 * i] = ((h & 0xffffu) >= thr16) ? v[2 * i] * scale : 0.f;
        v[2 * i + 1] = ((h >> 16) >= thr16) ? v[2 * i + 1] * scale : 0.f;
    }
}
template <int VEC>
__device__ __forceinline__ uint32_t dropout_mask16(uint32_t key, uint64_t e0, uint32_t thr16) {
    const uint32_t base = ((uint32_t)(e0 >> 1) ^ ((uint32_t)(e0 >> 33) * 0x9E3779B9U)) ^ key;
    uint32_t m = 0;
    if (VEC == 1) {
        const uint32_t h = lowbias32(base);
        return (((e0 & 1) ? (h >> 16) : (h & 0xffffu)) >= thr16) ? 1u : 0u;
    }
#pragma unroll
    for (int i = 0; i < VEC / 2; ++i) {
        const uint32_t h = lowbias32(base + (uint32_t)i);      // (e0 >> 1) + i: VEC consecutive elements, e0 % VEC == 0
        m |= ((h & 0xffffu) >= thr16 ? 1u : 0u) << (2 * i);
        m |= ((h >> 16) >= thr16 ? 1u : 0u) << (2 * i + 1);
    }
    return m;
}
// keep-mask for element index `e` (one Philox call covers 4 consecutive elements)
__device__ __forceinline__ bool dropout_keep(const uint64_t* rng, uint32_t layer, uint64_t e, float p) {
    uint64_t seed = rng[0], step = rng[1];
    uint4 r = philox4((uint32_t)seed, (uint32_t)(seed >> 32),
                      make_uint4((uint32_t)(e >> 2), (uint32_t)(e >> 34), (uint32_t)step, layer));
    uint32_t w = (e & 3) == 0 ? r.x : (e & 3) == 1 ? r.y : (e & 3) == 2 ? r.z : r.w;
    return (float)(w >> 8) * (1.0f / 16777216.0f) >= p;
}
