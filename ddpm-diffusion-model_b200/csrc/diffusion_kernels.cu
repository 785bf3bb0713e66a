// Diffusion-process elementwise kernels: q_sample, MSE fwd/bwd, DDPM / DDIM steps, image output,
// API-boundary layout conversion and the sinusoidal timestep embedding.
// Replaces the ATen chains of src/model/difussion_class.py:81-234 (46/76/118 launches per call in
// the reference, SURVEY.md §2.2 row 11) with one vectorised, coalesced launch each.  The ten [T]
// schedule tables live in __constant__ memory (40 KB for T=1000).
//
// HBM roofline (fp32 tensors): q_sample 12 B/elem, MSE 8 (6 with bf16 pred), DDPM step 16,
// DDIM step 12 (eta=0) / 16, to_image01 8.
#include "common.cuh"
#include <math.h>

int64_t g_ddpm_launches = 0;
extern "C" int ddpm_abi_struct_sizes(int32_t* out, int n) {
    const int32_t v[6] = {(int32_t)sizeof(ddpm_tensor), (int32_t)sizeof(ddpm_conv_args), (int32_t)sizeof(ddpm_lin_entry),
                          (int32_t)sizeof(ddpm_wgrad_args), (int32_t)sizeof(ddpm_pack_entry), (int32_t)sizeof(ddpm_adam_hyper)};
    int k = 0;
    for (; out && k < n && k < 6; ++k) out[k] = v[k];
    return k;
}

#define TMAX 1024
#define NTAB 10
__constant__ float c_tab[NTAB * TMAX];

struct Schedule {
    int T;
    int device;
    const float* dev;  // [10][T] copy owned by the caller (kept alive by the Diffusion module)
    uint64_t id;
};
static uint64_t g_next_id = 1;
static uint64_t g_const_owner[64] = {0};

extern "C" int ddpm_abi_version(void) { return 2; }

extern "C" int ddpm_num_sms(int device, int* out) {
    if (!out) return DDPM_E_ARG;
    CUDA_TRY(cudaDeviceGetAttribute(out, cudaDevAttrMultiProcessorCount, device));
    return 0;
}

extern "C" int64_t ddpm_launch_count(int reset) {
    int64_t v = g_ddpm_launches;
    if (reset) g_ddpm_launches = 0;
    return v;
}
extern "C" int ddpm_launch_count_add(int64_t n) { g_ddpm_launches += n; return 0; }

extern "C" int ddpm_schedule_create(const float* tables_dev, int T, int device, void** handle) {
    if (!tables_dev || !handle || T <= 0 || device < 0 || device >= 64) return DDPM_E_ARG;
    Schedule* s = new Schedule();
    s->T = T; s->device = device; s->dev = tables_dev; s->id = g_next_id++;
    *handle = s;
    return 0;
}

extern "C" int ddpm_schedule_destroy(void* handle) {
    if (!handle) return DDPM_E_ARG;
    Schedule* s = (Schedule*)handle;
    if (s->device >= 0 && s->device < 64 && g_const_owner[s->device] == s->id) g_const_owner[s->device] = 0;
    delete s;
    return 0;
}

// Make `s` the owner of the __constant__ bank on its device (stream-ordered D2D copy).
// Tables longer than TMAX are read from global memory instead.
static int bind_schedule(Schedule* s, cudaStream_t st, bool* use_const) {
    if (!s) return DDPM_E_NOTREADY;
    *use_const = s->T <= TMAX;
    if (!*use_const) return 0;
    if (g_const_owner[s->device] != s->id) {
        for (int r = 0; r < NTAB; ++r)
            CUDA_TRY(cudaMemcpyToSymbolAsync(c_tab, s->dev + (size_t)r * s->T, sizeof(float) * s->T,
                                             sizeof(float) * r * TMAX, cudaMemcpyDeviceToDevice, st));
        g_const_owner[s->device] = s->id;
    }
    return 0;
}

template <bool CONST> __device__ __forceinline__ float tab(const float* g, int T, int row, int t) {
    return CONST ? c_tab[row * TMAX + t] : g[(size_t)row * T + t];
}
__device__ __forceinline__ int clamp_t(int64_t t, int T) {
    return (int)(t < 0 ? 0 : (t > T - 1 ? T - 1 : t));
}

template <typename T> __device__ __forceinline__ float4 ld4(const T* p, int64_t i);
template <> __device__ __forceinline__ float4 ld4<float>(const float* p, int64_t i) {
    return *reinterpret_cast<const float4*>(p + i);
}
template <> __device__ __forceinline__ float4 ld4<bf16>(const bf16* p, int64_t i) {
    uint2 r = *reinterpret_cast<const uint2*>(p + i);
    float2 a = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&r.x));
    float2 b = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&r.y));
    return make_float4(a.x, a.y, b.x, b.y);
}
template <typename T> __device__ __forceinline__ void st4(T* p, int64_t i, float4 v);
template <> __device__ __forceinline__ void st4<float>(float* p, int64_t i, float4 v) {
    *reinterpret_cast<float4*>(p + i) = v;
}
template <> __device__ __forceinline__ void st4<bf16>(bf16* p, int64_t i, float4 v) {
    uint2 r;
    *reinterpret_cast<__nv_bfloat162*>(&r.x) = __floats2bfloat162_rn(v.x, v.y);
    *reinterpret_cast<__nv_bfloat162*>(&r.y) = __floats2bfloat162_rn(v.z, v.w);
    *reinterpret_cast<uint2*>(p + i) = r;
}

#define EW_THREADS 256
#define EW_UNROLL 4
#define EW_PER_BLOCK (EW_THREADS * EW_UNROLL * 4)

// Generic per-sample elementwise driver: F::coef(b) once per block, F::apply on float4 lanes.
// grid = (ceil(chw / EW_PER_BLOCK), B).  VEC=false is the scalar path for chw % 4 != 0.
template <typename F, bool VEC>
__global__ void __launch_bounds__(EW_THREADS) ew_kernel(F f, int64_t chw) {
    __shared__ typename F::Coef sc;
    const int b = blockIdx.y;
    if (threadIdx.x == 0) sc = f.coef(b);
    __syncthreads();
    const typename F::Coef c = sc;
    const int64_t base = (int64_t)b * chw;
    if (VEC) {
        int64_t i0 = ((int64_t)blockIdx.x * EW_THREADS * EW_UNROLL + threadIdx.x) * 4;
#pragma unroll
        for (int u = 0; u < EW_UNROLL; ++u) {
            int64_t i = i0 + (int64_t)u * EW_THREADS * 4;
            if (i < chw) f.apply4(c, base + i);
        }
    } else {
        int64_t i0 = (int64_t)blockIdx.x * EW_PER_BLOCK + threadIdx.x;
        for (int u = 0; u < EW_UNROLL * 4; ++u) {
            int64_t i = i0 + (int64_t)u * EW_THREADS;
            if (i < chw) f.apply1(c, base + i);
        }
    }
}

template <typename F> static int launch_ew(const F& f, int B, int64_t chw, bool aligned, cudaStream_t st) {
    if (B <= 0 || chw <= 0) return DDPM_E_ARG;
    dim3 grid(ceil_div(chw, EW_PER_BLOCK), B);
    if (aligned && (chw % 4) == 0) ew_kernel<F, true><<<grid, EW_THREADS, 0, st>>>(f, chw);
    else ew_kernel<F, false><<<grid, EW_THREADS, 0, st>>>(f, chw);
    LAUNCH_OK();
    return 0;
}
static inline bool al16(const void* p) { return (((uintptr_t)p) & 15) == 0; }
static inline bool al8(const void* p) { return (((uintptr_t)p) & 7) == 0; }

// ---------------------------------------------------------------- q_sample
template <bool CONST> struct QSample {
    const float* x0; const float* eps; const int64_t* t; float* xt; const float* g; int T;
    struct Coef { float a, s; };
    __device__ Coef coef(int b) const {
        int tt = clamp_t(t[b], T);
        return {tab<CONST>(g, T, 3, tt), tab<CONST>(g, T, 4, tt)};
    }
    __device__ __forceinline__ float f(const Coef& c, float x, float e) const {
        return __fadd_rn(__fmul_rn(c.a, x), __fmul_rn(c.s, e));   // torch: mul, mul, add (no FMA)
    }
    __device__ void apply4(const Coef& c, int64_t i) const {
        float4 x = ld4<float>(x0, i), e = ld4<float>(eps, i);
        st4<float>(xt, i, make_float4(f(c, x.x, e.x), f(c, x.y, e.y), f(c, x.z, e.z), f(c, x.w, e.w)));
    }
    __device__ void apply1(const Coef& c, int64_t i) const { xt[i] = f(c, x0[i], eps[i]); }
};

extern "C" int ddpm_q_sample(void* sched, const float* x0, const float* eps, const int64_t* t,
                             float* xt, int B, int64_t chw, void* stream) {
    if (!x0 || !eps || !t || !xt) return DDPM_E_ARG;
    Schedule* s = (Schedule*)sched; bool uc; cudaStream_t st = (cudaStream_t)stream;
    int rc = bind_schedule(s, st, &uc); if (rc) return rc;
    bool al = al16(x0) && al16(eps) && al16(xt);
    if (uc) { QSample<true> f{x0, eps, t, xt, s->dev, s->T}; return launch_ew(f, B, chw, al, st); }
    QSample<false> f{x0, eps, t, xt, s->dev, s->T}; return launch_ew(f, B, chw, al, st);
}

// ---------------------------------------------------------------- MSE forward / backward
template <typename TP, bool VEC>
__global__ void __launch_bounds__(EW_THREADS) mse_fwd_kernel(const TP* pred, const float* noise, const float* weight,
                                                             float* loss, int B, int64_t chw) {
    const int b = blockIdx.y;
    const int64_t base = (int64_t)b * chw;
    float acc = 0.f;
    if (VEC) {
        int64_t i0 = ((int64_t)blockIdx.x * EW_THREADS * EW_UNROLL + threadIdx.x) * 4;
#pragma unroll
        for (int u = 0; u < EW_UNROLL; ++u) {
            int64_t i = i0 + (int64_t)u * EW_THREADS * 4;
            if (i < chw) {
                float4 p = ld4<TP>(pred, base + i), n = ld4<float>(noise, base + i);
                float d0 = n.x - p.x, d1 = n.y - p.y, d2 = n.z - p.z, d3 = n.w - p.w;
                acc += d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
            }
        }
    } else {
        int64_t i0 = (int64_t)blockIdx.x * EW_PER_BLOCK + threadIdx.x;
        for (int u = 0; u < EW_UNROLL * 4; ++u) {
            int64_t i = i0 + (int64_t)u * EW_THREADS;
            if (i < chw) { float d = noise[base + i] - ldf<TP>(pred + base + i); acc += d * d; }
        }
    }
    __shared__ float red[EW_THREADS / 32];
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
        float v = threadIdx.x < EW_THREADS / 32 ? red[threadIdx.x] : 0.f;
        v = warp_sum(v);
        if (threadIdx.x == 0) {
            float w = weight ? weight[b] : 1.0f;
            atomicAdd(loss, v * (w / ((float)B * (float)chw)));
        }
    }
}

extern "C" int ddpm_mse_fwd(const void* pred, int pred_dtype, const float* noise, const float* weight,
                            float* loss, int B, int64_t chw, void* stream) {
    if (!pred || !noise || !loss || B <= 0 || chw <= 0) return DDPM_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid(ceil_div(chw, EW_PER_BLOCK), B);
    bool vec = (chw % 4) == 0 && al16(noise) && (pred_dtype == DDPM_F32 ? al16(pred) : al8(pred));
    if (pred_dtype == DDPM_F32) {
        if (vec) mse_fwd_kernel<float, true><<<grid, EW_THREADS, 0, st>>>((const float*)pred, noise, weight, loss, B, chw);
        else mse_fwd_kernel<float, false><<<grid, EW_THREADS, 0, st>>>((const float*)pred, noise, weight, loss, B, chw);
    } else if (pred_dtype == DDPM_BF16) {
        if (vec) mse_fwd_kernel<bf16, true><<<grid, EW_THREADS, 0, st>>>((const bf16*)pred, noise, weight, loss, B, chw);
        else mse_fwd_kernel<bf16, false><<<grid, EW_THREADS, 0, st>>>((const bf16*)pred, noise, weight, loss, B, chw);
    } else return DDPM_E_ARG;
    LAUNCH_OK();
    return 0;
}

template <typename TP> struct MseBwd {
    const TP* pred; const float* noise; const float* weight; const float* gout; TP* dpred; float inv;
    struct Coef { float k; };
    __device__ Coef coef(int b) const { return {2.0f * (weight ? weight[b] : 1.0f) * inv * gout[0]}; }
    __device__ void apply4(const Coef& c, int64_t i) const {
        float4 p = ld4<TP>(pred, i), n = ld4<float>(noise, i);
        st4<TP>(dpred, i, make_float4((p.x - n.x) * c.k, (p.y - n.y) * c.k, (p.z - n.z) * c.k, (p.w - n.w) * c.k));
    }
    __device__ void apply1(const Coef& c, int64_t i) const { stf<TP>(dpred + i, (ldf<TP>(pred + i) - noise[i]) * c.k); }
};

extern "C" int ddpm_mse_bwd(const void* pred, int pred_dtype, const float* noise, const float* weight,
                            const float* gout, void* dpred, int B, int64_t chw, void* stream) {
    if (!pred || !noise || !gout || !dpred || B <= 0 || chw <= 0) return DDPM_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    float inv = 1.0f / ((float)B * (float)chw);
    if (pred_dtype == DDPM_F32) {
        MseBwd<float> f{(const float*)pred, noise, weight, gout, (float*)dpred, inv};
        return launch_ew(f, B, chw, al16(pred) && al16(noise) && al16(dpred), st);
    } else if (pred_dtype == DDPM_BF16) {
        MseBwd<bf16> f{(const bf16*)pred, noise, weight, gout, (bf16*)dpred, inv};
        return launch_ew(f, B, chw, al8(pred) && al16(noise) && al8(dpred), st);
    }
    return DDPM_E_ARG;
}

// ---------------------------------------------------------------- x0_hat helpers
// x0_hat = (x_t - sqrt(1-ab) eps) / (sqrt(ab) + 1e-12), then dynamic threshold or clamp.
// a / b for a per-sample constant b with r = 1/b precomputed (IEEE) once per block: one Newton step on the
// quotient, 3 FP32 instructions, within 1 ulp of the correctly rounded quotient (IEEE division is ~12
// instructions and made the DDIM step instruction-bound: 67 % of HBM peak at eta = 0).
__device__ __forceinline__ float div_const(float a, float b, float r) {
    const float q = a * r;
    return fmaf(fmaf(-b, q, a), r, q);
}
struct X0Coef { float sa_eps, so, thr_div, r_sa, r_thr; int flags; };
__device__ __forceinline__ float x0_hat(const X0Coef& c, float x, float e) {
    float v = div_const(__fsub_rn(x, __fmul_rn(c.so, e)), c.sa_eps, c.r_sa);
    if (c.flags & DDPM_DYN_THRESH) { v = div_const(v, c.thr_div, c.r_thr); v = fminf(fmaxf(v, -1.f), 1.f); }
    else if (c.flags & DDPM_CLAMP_X0) v = fminf(fmaxf(v, -1.f), 1.f);
    return v;
}
template <bool CONST> __device__ __forceinline__ X0Coef make_x0coef(const float* g, int T, int tt, int flags,
                                                                     const float* amax, int b, float dyn_s) {
    X0Coef c;
    c.sa_eps = __fadd_rn(tab<CONST>(g, T, 3, tt), 1e-12f);
    c.so = tab<CONST>(g, T, 4, tt);
    c.flags = flags;
    c.thr_div = 1.f;
    if (flags & DDPM_DYN_THRESH) c.thr_div = fmaxf(fmaxf(amax[b], 1.0f), dyn_s);
    c.r_sa = __fdiv_rn(1.0f, c.sa_eps); c.r_thr = __fdiv_rn(1.0f, c.thr_div);
    return c;
}

template <typename TE, bool CONST> struct AbsMax {
    const float* xt; const TE* eps; const int64_t* t; float* amax; const float* g; int T;
};
template <typename TE, bool CONST>
__global__ void __launch_bounds__(EW_THREADS) absmax_kernel(AbsMax<TE, CONST> a, int64_t chw) {
    const int b = blockIdx.y;
    const int tt = clamp_t(a.t[b], a.T);
    X0Coef c = make_x0coef<CONST>(a.g, a.T, tt, 0, nullptr, b, 0.f);
    const int64_t base = (int64_t)b * chw;
    float m = 0.f;
    int64_t i0 = (int64_t)blockIdx.x * EW_PER_BLOCK + threadIdx.x;
    for (int u = 0; u < EW_UNROLL * 4; ++u) {
        int64_t i = i0 + (int64_t)u * EW_THREADS;
        if (i < chw) m = fmaxf(m, fabsf(x0_hat(c, a.xt[base + i], ldf<TE>(a.eps + base + i))));
    }
    m = warp_max(m);
    __shared__ float red[EW_THREADS / 32];
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x < 32) {
        float v = threadIdx.x < EW_THREADS / 32 ? red[threadIdx.x] : 0.f;
        v = warp_max(v);
        // non-negative floats order like their bit patterns
        if (threadIdx.x == 0) atomicMax(reinterpret_cast<int*>(a.amax + b), __float_as_int(v));
    }
}

extern "C" int ddpm_x0_absmax(void* sched, const float* xt, const void* eps, int eps_dtype,
                              const int64_t* t, float* amax, int B, int64_t chw, void* stream) {
    if (!xt || !eps || !t || !amax || B <= 0 || chw <= 0) return DDPM_E_ARG;
    Schedule* s = (Schedule*)sched; bool uc; cudaStream_t st = (cudaStream_t)stream;
    int rc = bind_schedule(s, st, &uc); if (rc) return rc;
    CUDA_TRY(cudaMemsetAsync(amax, 0, sizeof(float) * B, st));
    dim3 grid(ceil_div(chw, EW_PER_BLOCK), B);
#define GO(TE, CN) { AbsMax<TE, CN> a{xt, (const TE*)eps, t, amax, s->dev, s->T}; \
                     absmax_kernel<TE, CN><<<grid, EW_THREADS, 0, st>>>(a, chw); }
    if (eps_dtype == DDPM_F32) { if (uc) GO(float, true) else GO(float, false) }
    else if (eps_dtype == DDPM_BF16) { if (uc) GO(bf16, true) else GO(bf16, false) }
    else return DDPM_E_ARG;
#undef GO
    LAUNCH_OK();
    return 0;
}

// ---------------------------------------------------------------- DDPM ancestral step
template <typename TE, bool CONST> struct DdpmStep {
    const float* xt; const TE* eps; const float* noise; const int64_t* t; const float* amax; float dyn_s;
    int flags; float* out; const float* g; int T;
    struct Coef { X0Coef x; float c1, c2, sig; };
    __device__ Coef coef(int b) const {
        int64_t traw = t[b];
        int tt = clamp_t(traw, T);
        Coef c;
        c.x = make_x0coef<CONST>(g, T, tt, flags, amax, b, dyn_s);
        c.c1 = tab<CONST>(g, T, 8, tt);
        c.c2 = tab<CONST>(g, T, 9, tt);
        float nz = traw > 0 ? 1.f : 0.f;                                 // (t > 0).float()
        c.sig = __fmul_rn(nz, expf(__fmul_rn(0.5f, tab<CONST>(g, T, 7, tt))));
        return c;
    }
    __device__ __forceinline__ float f(const Coef& c, float x, float e, float z) const {
        float x0 = x0_hat(c.x, x, e);
        float mean = __fadd_rn(__fmul_rn(c.c1, x0), __fmul_rn(c.c2, x));
        return __fadd_rn(mean, __fmul_rn(c.sig, z));
    }
    __device__ void apply4(const Coef& c, int64_t i) const {
        float4 x = ld4<float>(xt, i), e = ld4<TE>(eps, i);
        float4 z = noise ? ld4<float>(noise, i) : make_float4(0.f, 0.f, 0.f, 0.f);
        st4<float>(out, i, make_float4(f(c, x.x, e.x, z.x), f(c, x.y, e.y, z.y), f(c, x.z, e.z, z.z), f(c, x.w, e.w, z.w)));
    }
    __device__ void apply1(const Coef& c, int64_t i) const {
        out[i] = f(c, xt[i], ldf<TE>(eps + i), noise ? noise[i] : 0.f);
    }
};

extern "C" int ddpm_p_sample_step(void* sched, const float* xt, const void* eps, int eps_dtype,
                                  const float* noise, const int64_t* t, const float* amax, float dyn_s,
                                  int flags, float* out, int B, int64_t chw, void* stream) {
    if (!xt || !eps || !t || !out) return DDPM_E_ARG;
    if ((flags & DDPM_DYN_THRESH) && !amax) return DDPM_E_ARG;
    Schedule* s = (Schedule*)sched; bool uc; cudaStream_t st = (cudaStream_t)stream;
    int rc = bind_schedule(s, st, &uc); if (rc) return rc;
    bool al = al16(xt) && al16(out) && (!noise || al16(noise)) && (eps_dtype == DDPM_F32 ? al16(eps) : al8(eps));
#define GO(TE, CN) { DdpmStep<TE, CN> f{xt, (const TE*)eps, noise, t, amax, dyn_s, flags, out, s->dev, s->T}; \
                     return launch_ew(f, B, chw, al, st); }
    if (eps_dtype == DDPM_F32) { if (uc) GO(float, true) else GO(float, false) }
    else if (eps_dtype == DDPM_BF16) { if (uc) GO(bf16, true) else GO(bf16, false) }
#undef GO
    return DDPM_E_ARG;
}

// ---------------------------------------------------------------- DDIM step
template <typename TE, bool CONST> struct DdimStep {
    const float* xt; const TE* eps; const float* noise; const int64_t* t; const int64_t* tp; float eta;
    const float* amax; float dyn_s; int flags; float* out; const float* g; int T;
    struct Coef { X0Coef x; float sq_at, inv_dir, r_dir, sq_ap, add, sigma; };
    __device__ Coef coef(int b) const {
        int tt = clamp_t(t[b], T), tq = clamp_t(tp[b], T);
        Coef c;
        c.x = make_x0coef<CONST>(g, T, tt, flags, amax, b, dyn_s);
        float a_t = tab<CONST>(g, T, 2, tt), a_p = tab<CONST>(g, T, 2, tq);
        float om = __fadd_rn(__fsub_rn(1.0f, a_t), 1e-12f);
        c.sq_at = sqrtf(a_t);
        c.inv_dir = sqrtf(om);                                          // divide by it (div_const), not multiply by 1/x
        c.r_dir = __fdiv_rn(1.0f, c.inv_dir);
        float s1 = sqrtf(__fdiv_rn(__fsub_rn(1.0f, a_p), om));
        float s2 = sqrtf(__fsub_rn(1.0f, __fdiv_rn(a_t, __fadd_rn(a_p, 1e-12f))));
        c.sigma = __fmul_rn(__fmul_rn(eta, s1), s2);
        c.sq_ap = sqrtf(a_p);
        c.add = sqrtf(fmaxf(__fsub_rn(__fsub_rn(1.0f, a_p), __fmul_rn(c.sigma, c.sigma)), 0.0f));
        return c;
    }
    __device__ __forceinline__ float f(const Coef& c, float x, float e, float z) const {
        float x0 = x0_hat(c.x, x, e);
        float dir = div_const(__fsub_rn(x, __fmul_rn(c.sq_at, x0)), c.inv_dir, c.r_dir);
        float r = __fadd_rn(__fmul_rn(c.sq_ap, x0), __fmul_rn(c.add, dir));
        return __fadd_rn(r, __fmul_rn(c.sigma, z));
    }
    __device__ void apply4(const Coef& c, int64_t i) const {
        float4 x = ld4<float>(xt, i), e = ld4<TE>(eps, i);
        float4 z = noise ? ld4<float>(noise, i) : make_float4(0.f, 0.f, 0.f, 0.f);
        st4<float>(out, i, make_float4(f(c, x.x, e.x, z.x), f(c, x.y, e.y, z.y), f(c, x.z, e.z, z.z), f(c, x.w, e.w, z.w)));
    }
    __device__ void apply1(const Coef& c, int64_t i) const {
        out[i] = f(c, xt[i], ldf<TE>(eps + i), noise ? noise[i] : 0.f);
    }
};

extern "C" int ddpm_ddim_step(void* sched, const float* xt, const void* eps, int eps_dtype,
                              const float* noise, const int64_t* t, const int64_t* t_prev, float eta,
                              const float* amax, float dyn_s, int flags, float* out, int B, int64_t chw,
                              void* stream) {
    if (!xt || !eps || !t || !t_prev || !out) return DDPM_E_ARG;
    if ((flags & DDPM_DYN_THRESH) && !amax) return DDPM_E_ARG;
    if (eta != 0.0f && !noise) return DDPM_E_ARG;
    Schedule* s = (Schedule*)sched; bool uc; cudaStream_t st = (cudaStream_t)stream;
    int rc = bind_schedule(s, st, &uc); if (rc) return rc;
    if (eta == 0.0f) noise = nullptr;   // sigma * z is exactly 0: skip the 4 B/elem read
    bool al = al16(xt) && al16(out) && (!noise || al16(noise)) && (eps_dtype == DDPM_F32 ? al16(eps) : al8(eps));
#define GO(TE, CN) { DdimStep<TE, CN> f{xt, (const TE*)eps, noise, t, t_prev, eta, amax, dyn_s, flags, out, s->dev, s->T}; \
                     return launch_ew(f, B, chw, al, st); }
    if (eps_dtype == DDPM_F32) { if (uc) GO(float, true) else GO(float, false) }
    else if (eps_dtype == DDPM_BF16) { if (uc) GO(bf16, true) else GO(bf16, false) }
#undef GO
    return DDPM_E_ARG;
}

// ---------------------------------------------------------------- to_image01
struct ToImg {
    const float* x; float* out;
    struct Coef { int dummy; };
    __device__ Coef coef(int) const { return {0}; }
    __device__ __forceinline__ static float f(float v) { return __fmul_rn(__fadd_rn(fminf(fmaxf(v, -1.f), 1.f), 1.0f), 0.5f); }
    __device__ void apply4(const Coef&, int64_t i) const {
        float4 v = ld4<float>(x, i);
        st4<float>(out, i, make_float4(f(v.x), f(v.y), f(v.z), f(v.w)));
    }
    __device__ void apply1(const Coef&, int64_t i) const { out[i] = f(x[i]); }
};
extern "C" int ddpm_to_image01(const float* x, float* out, int64_t n, void* stream) {
    if (!x || !out || n <= 0) return DDPM_E_ARG;
    ToImg f{x, out};
    return launch_ew(f, 1, n, al16(x) && al16(out), (cudaStream_t)stream);
}

// ---------------------------------------------------------------- image grid + uint8 (sampler output path)
// torchvision.utils.make_grid(padding, pad_value = 0) and save_image's `mul(255).add_(0.5).clamp_(0,255).to(uint8)` in
// one pass over the output pixels (ddpm_inference.py:41-45, ddpim_inference.py:90-93): the reference issues one
// narrow().copy_() launch per image plus four elementwise passes and a permute before the D2H copy.
__global__ void image_grid_kernel(const float* __restrict__ x, int N, int C, int H, int W, int xmaps, int pad, int Hg, int Wg,
                                  float* __restrict__ gf, uint8_t* __restrict__ gu) {
    const int64_t total = (int64_t)Hg * Wg;
    const int ch = H + pad, cw = W + pad;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int gy = (int)(i / Wg), gx = (int)(i - (int64_t)gy * Wg);
        int k = -1, iy = 0, ix = 0;
        if (N == 1) { k = 0; iy = gy; ix = gx; }                     // make_grid returns a single image unchanged
        else {
            const int y = gy - pad, x_ = gx - pad;
            if (y >= 0 && x_ >= 0) {
                const int cy = y / ch, cx = x_ / cw;
                iy = y - cy * ch; ix = x_ - cx * cw;
                if (iy < H && ix < W && cx < xmaps && cy * xmaps + cx < N) k = cy * xmaps + cx;
            }
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float v = k >= 0 ? x[(((int64_t)k * C + (C == 1 ? 0 : c)) * H + iy) * W + ix] : 0.f;
            if (gf) gf[(int64_t)c * total + i] = v;
            if (gu) gu[i * 3 + c] = (uint8_t)fminf(fmaxf(__fadd_rn(__fmul_rn(v, 255.f), 0.5f), 0.f), 255.f);
        }
    }
}
extern "C" int ddpm_image_grid(const float* x01, int N, int C, int H, int W, int nrow, int pad, float* grid_f32,
                               uint8_t* grid_u8, void* stream) {
    if (!x01 || N <= 0 || (C != 1 && C != 3) || H <= 0 || W <= 0 || nrow <= 0 || pad < 0 || (!grid_f32 && !grid_u8)) return DDPM_E_ARG;
    const int xmaps = nrow < N ? nrow : N, ymaps = (N + xmaps - 1) / xmaps;
    const int Hg = N == 1 ? H : (H + pad) * ymaps + pad, Wg = N == 1 ? W : (W + pad) * xmaps + pad;
    const int64_t total = (int64_t)Hg * Wg;
    int grid = (int)((total + 255) / 256); if (grid > 148 * 8) grid = 148 * 8;
    CUDA_TRY(launch_kernel(image_grid_kernel, dim3(grid), dim3(256), 0, (cudaStream_t)stream, x01, N, C, H, W, xmaps, pad, Hg, Wg,
                        grid_f32, grid_u8));
    LAUNCH_OK();
    return 0;
}

// ---------------------------------------------------------------- device-resident batch feeder (input side)
// ToTensor + Normalize([0.5]*3, [0.5]*3) of the reference's loaders (src/data/load_data_local.py:90-95,
// celebraHQ.py:40-43) applied to a uint8 NHWC dataset that lives in HBM: out[b][c][y][x] = (u8/255 - 0.5) / 0.5 for the
// sample idx[b], written as the NCHW fp32 batch `train_one_epoch` expects.  One thread per pixel (3 bytes in, three
// coalesced plane writes out); 3 B read + 12 B written per pixel.
__global__ void batch_from_u8_kernel(const uint8_t* __restrict__ data, const int64_t* __restrict__ idx, int B, int64_t hw,
                                     float* __restrict__ out) {
    const int64_t total = (int64_t)B * hw;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int b = (int)(i / hw); const int64_t p = i - (int64_t)b * hw;
        const uint8_t* src = data + ((int64_t)idx[b] * hw + p) * 3;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float t = __fdiv_rn((float)src[c], 255.f);                 // ToTensor
            out[((int64_t)b * 3 + c) * hw + p] = __fdiv_rn(__fsub_rn(t, 0.5f), 0.5f);   // Normalize(0.5, 0.5)
        }
    }
}
extern "C" int ddpm_batch_from_u8(const uint8_t* data, int64_t n_images, const int64_t* idx, int B, int H, int W, float* out,
                                  void* stream) {
    if (!data || !idx || !out || n_images <= 0 || B <= 0 || H <= 0 || W <= 0) return DDPM_E_ARG;
    const int64_t hw = (int64_t)H * W, total = (int64_t)B * hw;
    int grid = (int)((total + 255) / 256); if (grid > 148 * 16) grid = 148 * 16;
    CUDA_TRY(launch_kernel(batch_from_u8_kernel, dim3(grid), dim3(256), 0, (cudaStream_t)stream, data, idx, B, hw, out));
    LAUNCH_OK();
    return 0;
}

// ---------------------------------------------------------------- layout conversion
template <typename TS, typename TD, bool TO_NHWC>
__global__ void layout_kernel(char* nchw, int64_t sn, int64_t sc, int64_t sh, int64_t sw, TV v, int srcC) {
    int64_t total = (int64_t)v.N * v.H * v.W * v.C;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        int c = (int)(i % v.C); int64_t r = i / v.C;
        int x = (int)(r % v.W); r /= v.W;
        int y = (int)(r % v.H); int n = (int)(r / v.H);
        int64_t off = n * sn + c * sc + y * sh + x * sw;
        if (TO_NHWC) stf<TD>(v.at<TD>(n, y, x, c), c < srcC ? ldf<TS>(reinterpret_cast<const TS*>(nchw) + off) : 0.f);
        else stf<TD>(reinterpret_cast<TD*>(nchw) + off, ldf<TS>(v.at<TS>(n, y, x, c)));
    }
}

// Few channels (the API boundary: 3 image channels <-> a 16-channel padded NHWC tensor): one thread per PIXEL, so the
// NCHW side is read / written coalesced along x and the NHWC side as one contiguous run per thread (the per-element
// kernel above walks c fastest: plane-strided 4-byte accesses and three integer divisions per element -- 33 us for a 6 MB
// tensor, twice per UNet evaluation).
template <typename TS, typename TD, bool TO_NHWC>
__global__ void layout_pix_kernel(char* nchw, int64_t sn, int64_t sc, int64_t sh, int64_t sw, TV v, int srcC) {
    const int64_t total = (int64_t)v.N * v.H * v.W;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int x = (int)(i % v.W); const int64_t r = i / v.W;
        const int y = (int)(r % v.H), n = (int)(r / v.H);
        const int64_t base = n * sn + y * sh + x * sw;
        if (TO_NHWC) {
            TD* d = v.at<TD>(n, y, x, 0);
            const TS* sp = reinterpret_cast<const TS*>(nchw) + base;
            for (int c0 = 0; c0 < v.C; c0 += 8) {
                float f[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) f[j] = (c0 + j < srcC) ? ldf<TS>(sp + (int64_t)(c0 + j) * sc) : 0.f;
                if (sizeof(TD) == 2 && c0 + 8 <= v.C && ((uintptr_t)(d + c0) & 15) == 0) {
                    uint4 o; __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
                    for (int j = 0; j < 4; ++j) h[j] = __floats2bfloat162_rn(f[2 * j], f[2 * j + 1]);
                    *reinterpret_cast<uint4*>(d + c0) = o;
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j) if (c0 + j < v.C) stf<TD>(d + c0 + j, f[j]);
                }
            }
        } else {
            const TS* sp = v.at<TS>(n, y, x, 0);
            TD* d = reinterpret_cast<TD*>(nchw) + base;
            for (int c = 0; c < v.C; ++c) stf<TD>(d + (int64_t)c * sc, ldf<TS>(sp + c));
        }
    }
}
#define LAYOUT_GO(TS, TD, DIR, PTR, SRCC) { \
        if (v.C <= 32) { \
            const int64_t px = (int64_t)v.N * v.H * v.W; int g = (int)((px + 255) / 256); if (g > 148 * 16) g = 148 * 16; \
            CUDA_TRY(launch_kernel(layout_pix_kernel<TS, TD, DIR>, dim3(g), dim3(256), 0, st, PTR, sn, sc, sh, sw, v, SRCC)); \
        } else layout_kernel<TS, TD, DIR><<<grid, 256, 0, st>>>(PTR, sn, sc, sh, sw, v, SRCC); }

extern "C" int ddpm_nchw_to_nhwc(const void* src, int src_dtype, int src_C, int64_t sn, int64_t sc, int64_t sh,
                                 int64_t sw, const ddpm_tensor* dst, int dst_dtype, void* stream) {
    if (!src || !tensor_ok(dst) || src_C <= 0 || src_C > dst->C) return DDPM_E_ARG;
    const int srcC = src_C;
    TV v(*dst); cudaStream_t st = (cudaStream_t)stream;
    int64_t total = (int64_t)v.N * v.H * v.W * v.C;
    int grid = (int)((total + 255) / 256); if (grid > 148 * 16) grid = 148 * 16;
    char* s = (char*)src;
    if (src_dtype == DDPM_F32 && dst_dtype == DDPM_F32) LAYOUT_GO(float, float, true, s, srcC)
    else if (src_dtype == DDPM_F32 && dst_dtype == DDPM_BF16) LAYOUT_GO(float, bf16, true, s, srcC)
    else if (src_dtype == DDPM_BF16 && dst_dtype == DDPM_BF16) LAYOUT_GO(bf16, bf16, true, s, srcC)
    else if (src_dtype == DDPM_BF16 && dst_dtype == DDPM_F32) LAYOUT_GO(bf16, float, true, s, srcC)
    else return DDPM_E_ARG;
    LAUNCH_OK();
    return 0;
}

extern "C" int ddpm_nhwc_to_nchw(const ddpm_tensor* src, int src_dtype, void* dst, int dst_dtype, int64_t sn,
                                 int64_t sc, int64_t sh, int64_t sw, void* stream) {
    if (!dst || !tensor_ok(src)) return DDPM_E_ARG;
    TV v(*src); cudaStream_t st = (cudaStream_t)stream;
    int64_t total = (int64_t)v.N * v.H * v.W * v.C;
    int grid = (int)((total + 255) / 256); if (grid > 148 * 16) grid = 148 * 16;
    char* d = (char*)dst;
    if (src_dtype == DDPM_F32 && dst_dtype == DDPM_F32) LAYOUT_GO(float, float, false, d, v.C)
    else if (src_dtype == DDPM_BF16 && dst_dtype == DDPM_F32) LAYOUT_GO(bf16, float, false, d, v.C)
    else if (src_dtype == DDPM_BF16 && dst_dtype == DDPM_BF16) LAYOUT_GO(bf16, bf16, false, d, v.C)
    else if (src_dtype == DDPM_F32 && dst_dtype == DDPM_BF16) LAYOUT_GO(float, bf16, false, d, v.C)
    else return DDPM_E_ARG;
    LAUNCH_OK();
    return 0;
}

// ---------------------------------------------------------------- sinusoidal embedding
// attention.py:13-22: freq_i = exp(-ln(1e4)/(half-1) * i); [sin(t f) | cos(t f)] (+ zero pad if odd)
template <typename TD>
__global__ void sinusoid_kernel(const void* t, int t_is_float, int B, int dim, TD* out) {
    int half = dim / 2;
    float k = logf(10000.0f) / (float)(half - 1);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < B * dim; i += gridDim.x * blockDim.x) {
        int b = i / dim, j = i % dim;
        float tv = t_is_float ? ((const float*)t)[b] : (float)((const int64_t*)t)[b];
        float r = 0.f;
        if (j < 2 * half) {
            int jj = j < half ? j : j - half;
            float ang = __fmul_rn(tv, expf(__fmul_rn((float)jj, -k)));
            r = j < half ? sinf(ang) : cosf(ang);
        }
        stf<TD>(out + i, r);
    }
}
extern "C" int ddpm_sinusoid(const void* t, int t_is_float, int B, int dim, void* out, int dtype, void* stream) {
    if (!t || !out || B <= 0 || dim < 4) return DDPM_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    int grid = ceil_div((int64_t)B * dim, 256);
    if (dtype == DDPM_F32) sinusoid_kernel<float><<<grid, 256, 0, st>>>(t, t_is_float, B, dim, (float*)out);
    else if (dtype == DDPM_BF16) sinusoid_kernel<bf16><<<grid, 256, 0, st>>>(t, t_is_float, B, dim, (bf16*)out);
    else return DDPM_E_ARG;
    LAUNCH_OK();
    return 0;
}
