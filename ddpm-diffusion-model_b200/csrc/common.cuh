// Shared device/host helpers for libddpm_b200 (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <type_traits>
#include "../../include/ddpm_b200.h"

typedef __nv_bfloat16 bf16;
typedef __half f16;

// The two 16-bit activation formats (DDPM_BF16, DDPM_F16): everything a kernel needs to know about one.  Kernels take the
// element type as a template parameter and read the format from here.  fp32 -> 16-bit conversions round to nearest; for
// fp16 that gives +-inf beyond 65504 (IEEE, no saturation), which is what a GradScaler relies on to detect overflow.
template <typename T> struct Fmt16;
template <> struct Fmt16<bf16> {
    typedef __nv_bfloat162 T2;
    static constexpr CUtensorMapDataType tma_type = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    static constexpr uint32_t idesc_ab = (1u << 7) | (1u << 10);   // tcgen05.mma kind::f16: A and B format BF16 (bits 7-9, 10-12)
    static constexpr uint16_t one = 0x3F80;                         // 1.0
    __device__ __forceinline__ static float to_f(bf16 h) { return __bfloat162float(h); }
    __device__ __forceinline__ static bf16 from_f(float v) { return __float2bfloat16_rn(v); }
    __device__ __forceinline__ static float2 to_f2(T2 h) { return __bfloat1622float2(h); }
    __device__ __forceinline__ static T2 from_f2(float a, float b) { return __floats2bfloat162_rn(a, b); }
    // the two elements of a 32-bit word in one integer instruction each (a bf16 is the upper half of an fp32)
    __device__ __forceinline__ static void unpack(uint32_t w, float& lo, float& hi) {
        lo = __uint_as_float(w << 16); hi = __uint_as_float(w & 0xffff0000u);
    }
};
template <> struct Fmt16<f16> {
    typedef __half2 T2;
    static constexpr CUtensorMapDataType tma_type = CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    static constexpr uint32_t idesc_ab = 0u;                        // A and B format F16
    static constexpr uint16_t one = 0x3C00;
    __device__ __forceinline__ static float to_f(f16 h) { return __half2float(h); }
    __device__ __forceinline__ static f16 from_f(float v) { return __float2half_rn(v); }
    __device__ __forceinline__ static float2 to_f2(T2 h) { return __half22float2(h); }
    __device__ __forceinline__ static T2 from_f2(float a, float b) { return __floats2half2_rn(a, b); }
    __device__ __forceinline__ static void unpack(uint32_t w, float& lo, float& hi) {
        const float2 f = __half22float2(*reinterpret_cast<const T2*>(&w));
        lo = f.x; hi = f.y;
    }
};
// 2-wide access through a 32-bit word (the element pair of a uint2 / uint4 lane)
template <typename T> __device__ __forceinline__ float2 unpack2(const uint32_t& w) {
    return Fmt16<T>::to_f2(*reinterpret_cast<const typename Fmt16<T>::T2*>(&w));
}
template <typename T> __device__ __forceinline__ void pack2(uint32_t& w, float a, float b) {
    *reinterpret_cast<typename Fmt16<T>::T2*>(&w) = Fmt16<T>::from_f2(a, b);
}

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
    __device__ __forceinline__ static float ld(const bf16* p) { return Fmt16<bf16>::to_f(*p); }
    __device__ __forceinline__ static void st(bf16* p, float v) { *p = Fmt16<bf16>::from_f(v); }
};
template <> struct Cvt<f16> {
    __device__ __forceinline__ static float ld(const f16* p) { return Fmt16<f16>::to_f(*p); }
    __device__ __forceinline__ static void st(f16* p, float v) { *p = Fmt16<f16>::from_f(v); }
};
template <typename T> __device__ __forceinline__ float ldf(const T* p) { return Cvt<T>::ld(p); }
template <typename T> __device__ __forceinline__ void stf(T* p, float v) { Cvt<T>::st(p, v); }

// 8-element (bf16 / fp16) / 4-element (fp32) 16-byte vectors of activations
template <typename T> struct Vec16 {
    static constexpr int N = 8;
    float v[8];
    __device__ __forceinline__ void load(const T* p) {
        uint4 t = *reinterpret_cast<const uint4*>(p);
        const typename Fmt16<T>::T2* h = reinterpret_cast<const typename Fmt16<T>::T2*>(&t);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            float2 f = Fmt16<T>::to_f2(h[i]);
            v[2 * i] = f.x; v[2 * i + 1] = f.y;
        }
    }
    __device__ __forceinline__ void store(T* p) const {
        uint4 t;
        typename Fmt16<T>::T2* h = reinterpret_cast<typename Fmt16<T>::T2*>(&t);
#pragma unroll
        for (int i = 0; i < 4; ++i) h[i] = Fmt16<T>::from_f2(v[2 * i], v[2 * i + 1]);
        *reinterpret_cast<uint4*>(p) = t;
    }
};
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
// <= |z| * 2.5e-4 -- below the bf16 resolution of the tensors these kernels write; the fp32 kernels keep silu_f, and so do
// the fp16 ones: fp16 has 3 more significant bits, and where SiLU cancels (silu(-3) = -0.14, silu(-6) = -0.015) that bound
// is ~5 and ~200 fp16 ulps of the result.
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

// Dropout keep-bits.  The GroupNorm kernels are instruction-bound on B200 (an SM has ~22 B/clk of HBM
// bandwidth, i.e. a budget of ~20 instructions per bf16 element), and Philox4x32-10 cost ~12 of them.
// Parity with ATen's mask is statistical only (SURVEY.md §7), so the mask comes from a counter hash.  Element e
// belongs to the 32-bit word w = e >> 1 and uses 16-bit half (e & 1) of lowbias32(((w & ~3) ^ key) + (w & 3)),
// key = dropout_key(seed, step, layer); keep iff half >= thr16 = (uint32_t)(p * 65536 + 0.5).  e is the logical NHWC
// index ((n*H + y)*W + x)*C + c of the view, wrapped to 32 bits: it does not depend on the pitch, the halo or the
// channel offset of the buffer.  The hash input is a bijection of w for every key (the low two bits of w are added
// to a block base whose low bits are key & 3, so no two words share an input), and it is what the bf16 path, which
// training runs, draws with one XOR per 8-element packet.  ~4 instructions per element; fp32 (VEC 4), bf16 (VEC 8)
// and scalar paths draw the same mask, so forward and backward may take different paths and still recompute the
// same mask from (seed, step, layer, index).
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
// (e0 % VEC == 0 for VEC > 1).  For VEC 8 the packet's four words are one aligned block (w0 & 3 == 0), so the block
// base is w0 ^ key; VEC 4 covers half a block and the scalar path one word, so they add w & 3 themselves.
template <int VEC>
__device__ __forceinline__ void dropout_apply(float* v, uint32_t key, uint32_t e0, uint32_t thr16, float scale) {
    const uint32_t w0 = e0 >> 1;
    const uint32_t base = VEC == 8 ? (w0 ^ key) : ((w0 & ~3u) ^ key) + (w0 & 3u);
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
