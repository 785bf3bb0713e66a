// Optimiser-side parameter pass over flat fp32 arenas.
// Replaces scaler.unscale_ + clip_grad_norm_ + AdamW.step + EMA.update
// (src/training_loops/train_one_epoch.py:94-115, src/training_loops/ema.py:15-23; 1,274 ATen calls
// per update in the reference, SURVEY.md §2.2 row 12) with one reduction and one fused update.
//
// HBM roofline: reduce 4 B/param; update reads g,p,m,v,ema (20 B) and writes p,m,v,ema (16 B)
// = 40 B/param in total.
#include "common.cuh"
#include <math.h>

#define PT 256
#define PU 4   // float4 per thread per iteration

// stats[0] += sum g^2 ; stats[1] = 1 if any non-finite
__global__ void __launch_bounds__(PT) param_reduce_kernel(const float* __restrict__ g, int64_t n, float* stats) {
    float acc = 0.f; int bad = 0;
    const int64_t n4 = n >> 2;
    const float4* g4 = reinterpret_cast<const float4*>(g);
    for (int64_t i = (int64_t)blockIdx.x * PT + threadIdx.x; i < n4; i += (int64_t)gridDim.x * PT) {
        float4 v = g4[i];
        acc += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
        bad |= !(isfinite(v.x) && isfinite(v.y) && isfinite(v.z) && isfinite(v.w));
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
        float v = g[(n4 << 2) + threadIdx.x]; acc += v * v; bad |= !isfinite(v);
    }
    acc = warp_sum(acc);
    bad = __any_sync(0xffffffffu, bad);
    __shared__ float red[PT / 32]; __shared__ int sbad;
    if (threadIdx.x == 0) sbad = 0;
    __syncthreads();
    if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5] = acc; if (bad) sbad = 1; }
    __syncthreads();
    if (threadIdx.x < 32) {
        float v = threadIdx.x < PT / 32 ? red[threadIdx.x] : 0.f;
        v = warp_sum(v);
        if (threadIdx.x == 0) {
            atomicAdd(&stats[0], v);
            if (sbad || !isfinite(v)) stats[1] = 1.0f;
        }
    }
}

extern "C" int ddpm_param_reduce(const float* grad, int64_t n, float* stats, void* stream) {
    if (!grad || !stats || n <= 0 || (((uintptr_t)grad) & 15)) return DDPM_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemsetAsync(stats, 0, sizeof(float) * 4, st));
    int grid = (int)(((n >> 2) + PT * PU - 1) / (PT * PU));
    if (grid > 148 * 8) grid = 148 * 8;
    if (grid < 1) grid = 1;
    param_reduce_kernel<<<grid, PT, 0, st>>>(grad, n, stats);
    LAUNCH_OK();
    return 0;
}

struct UpdCoef { float gmul, lr, b1, b2, eps, wd, bc1, rsqrt_bc2, decay; int skip, adamw; };

__device__ __forceinline__ void adam_elem(const UpdCoef& c, float& p, float g, float& m, float& v) {
    g *= c.gmul;
    if (c.adamw) p *= (1.0f - c.lr * c.wd); else g = fmaf(c.wd, p, g);
    m = fmaf(g - m, 1.0f - c.b1, m);                       // exp_avg.lerp_(grad, 1-beta1)
    v = fmaf(c.b2, v, (1.0f - c.b2) * g * g);
    float denom = sqrtf(v) * c.rsqrt_bc2 + c.eps;
    p -= (c.lr / c.bc1) * (m / denom);
}

__global__ void __launch_bounds__(PT) param_update_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                          float* __restrict__ m, float* __restrict__ v,
                                                          float* __restrict__ ema, int64_t n, const float* stats,
                                                          const float* step_p, const float* scale_p, ddpm_adam_hyper h) {
    UpdCoef c;
    {
        float scale = scale_p ? scale_p[0] : 1.0f;
        float inv = scale > 0.f ? 1.0f / scale : 1.0f;
        c.skip = stats[1] != 0.0f;
        float gnorm = sqrtf(stats[0]) * inv;                // norm of the unscaled gradient
        float clip = 1.0f;
        if (h.max_norm > 0.f) clip = fminf(h.max_norm / (gnorm + 1e-6f), 1.0f);
        c.gmul = inv * clip;
        float step = step_p[0] + 1.0f;                      // 1-based step of this update
        c.lr = h.lr; c.b1 = h.beta1; c.b2 = h.beta2; c.eps = h.eps; c.wd = h.weight_decay;
        c.bc1 = 1.0f - powf(h.beta1, step);
        c.rsqrt_bc2 = rsqrtf(1.0f - powf(h.beta2, step));
        c.decay = h.ema_decay; c.adamw = h.adamw;
    }
    const int64_t n4 = n >> 2;
    float4* p4 = reinterpret_cast<float4*>(p); const float4* g4 = reinterpret_cast<const float4*>(g);
    float4* m4 = reinterpret_cast<float4*>(m); float4* v4 = reinterpret_cast<float4*>(v);
    float4* e4 = reinterpret_cast<float4*>(ema);
    const float od = 1.0f - c.decay;
    for (int64_t i = (int64_t)blockIdx.x * PT + threadIdx.x; i < n4; i += (int64_t)gridDim.x * PT) {
        float4 pp = p4[i];
        if (!c.skip) {
            float4 gg = g4[i], mm = m4[i], vv = v4[i];
            adam_elem(c, pp.x, gg.x, mm.x, vv.x); adam_elem(c, pp.y, gg.y, mm.y, vv.y);
            adam_elem(c, pp.z, gg.z, mm.z, vv.z); adam_elem(c, pp.w, gg.w, mm.w, vv.w);
            p4[i] = pp; m4[i] = mm; v4[i] = vv;
        }
        if (ema) {
            float4 ee = e4[i];
            ee.x = fmaf(ee.x, c.decay, od * pp.x); ee.y = fmaf(ee.y, c.decay, od * pp.y);
            ee.z = fmaf(ee.z, c.decay, od * pp.z); ee.w = fmaf(ee.w, c.decay, od * pp.w);
            e4[i] = ee;
        }
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
        int64_t i = (n4 << 2) + threadIdx.x;
        float pp = p[i];
        if (!c.skip) { float mm = m[i], vv = v[i]; adam_elem(c, pp, g[i], mm, vv); p[i] = pp; m[i] = mm; v[i] = vv; }
        if (ema) ema[i] = fmaf(ema[i], c.decay, od * pp);
    }
}

__global__ void step_bump_kernel(float* step, const float* stats) {
    if (stats[1] == 0.0f) step[0] += 1.0f;
}

extern "C" int ddpm_param_update(float* p, const float* g, float* m, float* v, float* ema, int64_t n,
                                 const float* stats, float* step, const float* scale, const ddpm_adam_hyper* h,
                                 void* stream) {
    if (!p || !g || !m || !v || !stats || !step || !h || n <= 0) return DDPM_E_ARG;
    if ((((uintptr_t)p) | ((uintptr_t)g) | ((uintptr_t)m) | ((uintptr_t)v) | ((uintptr_t)ema)) & 15) return DDPM_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    int grid = (int)(((n >> 2) + PT * PU - 1) / (PT * PU));
    if (grid > 148 * 8) grid = 148 * 8;
    if (grid < 1) grid = 1;
    param_update_kernel<<<grid, PT, 0, st>>>(p, g, m, v, ema, n, stats, step, scale, *h);
    LAUNCH_OK();
    step_bump_kernel<<<1, 1, 0, st>>>(step, stats);
    LAUNCH_OK();
    return 0;
}

// torch.amp.GradScaler.update (_amp_update_scale_) on the scaler's own _scale / _growth_tracker tensors
// stats[2] <- the scale this step's gradients carried (read by the host-side grad-norm diagnostic AFTER the update)
__global__ void scaler_update_kernel(float* scale, int* tracker, float* stats, float growth, float backoff, int interval) {
    stats[2] = scale[0];
    if (stats[1] != 0.0f) { scale[0] *= backoff; tracker[0] = 0; }
    else {
        int t = tracker[0] + 1;
        if (t >= interval) { float ns = scale[0] * growth; if (isfinite(ns)) scale[0] = ns; t = 0; }
        tracker[0] = t;
    }
}
extern "C" int ddpm_scaler_update(float* scale, int32_t* tracker, float* stats, float growth, float backoff,
                                  int interval, void* stream) {
    if (!scale || !tracker || !stats || interval <= 0) return DDPM_E_ARG;
    scaler_update_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(scale, tracker, stats, growth, backoff, interval);
    LAUNCH_OK();
    return 0;
}

// unscale + clip in place for optimisers other than Adam(W): g *= clip/scale (0 when inf was found)
__global__ void __launch_bounds__(PT) grad_scale_kernel(float* __restrict__ g, int64_t n, const float* stats,
                                                        const float* scale_p, float max_norm) {
    float scale = scale_p ? scale_p[0] : 1.0f;
    float inv = scale > 0.f ? 1.0f / scale : 1.0f;
    float mul = inv;
    if (max_norm > 0.f) mul *= fminf(max_norm / (sqrtf(stats[0]) * inv + 1e-6f), 1.0f);
    if (stats[1] != 0.0f) mul = 0.f;
    for (int64_t i = (int64_t)blockIdx.x * PT + threadIdx.x; i < n; i += (int64_t)gridDim.x * PT) g[i] *= mul;
}
extern "C" int ddpm_grad_unscale_clip(float* g, int64_t n, const float* stats, const float* scale, float max_norm,
                                      void* stream) {
    if (!g || !stats || n <= 0) return DDPM_E_ARG;
    int grid = (int)((n + PT * 4 - 1) / (PT * 4));
    if (grid > 148 * 8) grid = 148 * 8;
    grad_scale_kernel<<<grid, PT, 0, (cudaStream_t)stream>>>(g, n, stats, scale, max_norm);
    LAUNCH_OK();
    return 0;
}

__global__ void __launch_bounds__(PT) ema_kernel(float* __restrict__ s, const float* __restrict__ p, int64_t n, float d) {
    const float od = 1.0f - d;
    const int64_t n4 = n >> 2;
    float4* s4 = reinterpret_cast<float4*>(s); const float4* p4 = reinterpret_cast<const float4*>(p);
    for (int64_t i = (int64_t)blockIdx.x * PT + threadIdx.x; i < n4; i += (int64_t)gridDim.x * PT) {
        float4 a = s4[i], b = p4[i];
        // shadow.mul_(d).add_(p, alpha=1-d): round(round(s*d) + (1-d)*p) -> fma on the second term
        a.x = fmaf(od, b.x, __fmul_rn(a.x, d)); a.y = fmaf(od, b.y, __fmul_rn(a.y, d));
        a.z = fmaf(od, b.z, __fmul_rn(a.z, d)); a.w = fmaf(od, b.w, __fmul_rn(a.w, d));
        s4[i] = a;
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
        int64_t i = (n4 << 2) + threadIdx.x;
        s[i] = fmaf(od, p[i], __fmul_rn(s[i], d));
    }
}
extern "C" int ddpm_ema_update(float* shadow, const float* p, int64_t n, float decay, void* stream) {
    if (!shadow || !p || n <= 0 || ((((uintptr_t)shadow) | ((uintptr_t)p)) & 15)) return DDPM_E_ARG;
    int grid = (int)(((n >> 2) + PT * PU - 1) / (PT * PU));
    if (grid > 148 * 8) grid = 148 * 8;
    if (grid < 1) grid = 1;
    ema_kernel<<<grid, PT, 0, (cudaStream_t)stream>>>(shadow, p, n, decay);
    LAUNCH_OK();
    return 0;
}

__global__ void rng_advance_kernel(uint64_t* rng) { rng[1] += 1; }
extern "C" int ddpm_rng_advance(uint64_t* rng, void* stream) {
    if (!rng) return DDPM_E_ARG;
    rng_advance_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(rng);
    LAUNCH_OK();
    return 0;
}

// ------------------------------------------------------------------------------------ weight packing
// OIHW fp32 -> fwd [CoP][tap][CiP] and dgrad [CiP][KH*KW-1-tap][CoP] in the activation dtype (zero padded).
template <typename T>
__global__ void pack_kernel(const float* __restrict__ w, int Cout, int Cin, int KH, int KW, int CiP, int CoP, T* wf, T* wd) {
    const int taps = KH * KW;
    const int64_t total = (int64_t)CoP * CiP * taps;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        // i enumerates the fwd layout (coalesced writes): co, tap, ci
        int ci = (int)(i % CiP); int64_t r = i / CiP;
        int tap = (int)(r % taps); int co = (int)(r / taps);
        float v = (ci < Cin && co < Cout) ? w[((int64_t)co * Cin + ci) * taps + tap] : 0.f;
        if (wf) stf<T>(wf + i, v);
        if (wd) stf<T>(wd + ((int64_t)ci * taps + (taps - 1 - tap)) * CoP + co, v);
    }
}
extern "C" int ddpm_pack_weights(const float* w, int Cout, int Cin, int KH, int KW, void* w_fwd, void* w_dgrad,
                                 int dtype, int cin_pad, int cout_pad, void* stream) {
    if (!w || (!w_fwd && !w_dgrad) || Cout <= 0 || Cin <= 0 || KH <= 0 || KW <= 0) return DDPM_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    int CiP = cin_pad > 0 ? cin_pad : Cin, CoP = cout_pad > 0 ? cout_pad : Cout;
    if (CiP < Cin || CoP < Cout) return DDPM_E_ARG;
    int64_t total = (int64_t)CoP * CiP * KH * KW;
    int grid = (int)((total + 255) / 256); if (grid > 148 * 8) grid = 148 * 8;
    if (dtype == DDPM_F32) pack_kernel<float><<<grid, 256, 0, st>>>(w, Cout, Cin, KH, KW, CiP, CoP, (float*)w_fwd, (float*)w_dgrad);
    else if (dtype == DDPM_BF16) pack_kernel<bf16><<<grid, 256, 0, st>>>(w, Cout, Cin, KH, KW, CiP, CoP, (bf16*)w_fwd, (bf16*)w_dgrad);
    else if (dtype == DDPM_F16) pack_kernel<f16><<<grid, 256, 0, st>>>(w, Cout, Cin, KH, KW, CiP, CoP, (f16*)w_fwd, (f16*)w_dgrad);
    else return DDPM_E_ARG;
    LAUNCH_OK();
    return 0;
}

// Phase weights of conv3x3(nearest_upsample_x2(x)) evaluated on the low-resolution x (see DDPM_CONV_UP2X_PHASE):
// rows (py, ty) -> which ky of the 3x3 filter land on low-res row y + ty + py - 1.
template <typename T>
__global__ void pack_up2x_kernel(const float* __restrict__ w, int Cout, int Cin, T* out) {
    const int64_t total = (int64_t)4 * Cout * 4 * Cin;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        int ci = (int)(i % Cin); int64_t r = i / Cin;
        int t = (int)(r % 4); r /= 4;
        int co = (int)(r % Cout); int ph = (int)(r / Cout);
        const int py = ph >> 1, px = ph & 1, ty = t >> 1, tx = t & 1;
        // S(0,0)={0}, S(0,1)={1,2}, S(1,0)={0,1}, S(1,1)={2}
        const int ky0 = (py == 0) ? (ty == 0 ? 0 : 1) : (ty == 0 ? 0 : 2), ky1 = (py == 0) ? (ty == 0 ? 0 : 2) : (ty == 0 ? 1 : 2);
        const int kx0 = (px == 0) ? (tx == 0 ? 0 : 1) : (tx == 0 ? 0 : 2), kx1 = (px == 0) ? (tx == 0 ? 0 : 2) : (tx == 0 ? 1 : 2);
        const float* wk = w + ((int64_t)co * Cin + ci) * 9;
        float v = 0.f;
        for (int ky = ky0; ky <= ky1; ++ky)
            for (int kx = kx0; kx <= kx1; ++kx) v += wk[ky * 3 + kx];
        stf<T>(out + i, v);
    }
}
extern "C" int ddpm_pack_weights_up2x(const float* w, int Cout, int Cin, void* out, int dtype, void* stream) {
    if (!w || !out || Cout <= 0 || Cin <= 0) return DDPM_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    int64_t total = (int64_t)16 * Cout * Cin;
    int grid = (int)((total + 255) / 256); if (grid > 148 * 8) grid = 148 * 8;
    if (dtype == DDPM_F32) pack_up2x_kernel<float><<<grid, 256, 0, st>>>(w, Cout, Cin, (float*)out);
    else if (dtype == DDPM_BF16) pack_up2x_kernel<bf16><<<grid, 256, 0, st>>>(w, Cout, Cin, (bf16*)out);
    else if (dtype == DDPM_F16) pack_up2x_kernel<f16><<<grid, 256, 0, st>>>(w, Cout, Cin, (f16*)out);
    else return DDPM_E_ARG;
    LAUNCH_OK();
    return 0;
}

// All packed copies in ONE launch (after the optimiser step every weight is stale at once; 76 per-weight launches
// of a few microseconds each were 0.4 ms of a 16 ms step).  `entries` lives in device memory.
// Tiles of 32 output x 32 input channels (x all taps) go through shared memory: the OIHW rows are read fully coalesced
// (32*taps contiguous floats per output channel) and both packed layouts are written in 64-byte runs -- the element-wise
// version read with a stride of `taps` floats and scattered the dgrad copy two bytes at a time (139 us for 100 MB).
#define PK_T 32
// the entries live in device memory, so an unknown dtype code cannot be refused by the call: its copies are not written
__device__ __forceinline__ void pack_store(void* dst, int dtype, int64_t o, float v) {
    if (dtype == DDPM_BF16) stf<bf16>((bf16*)dst + o, v);
    else if (dtype == DDPM_F16) stf<f16>((f16*)dst + o, v);
    else if (dtype == DDPM_F32) ((float*)dst)[o] = v;
}
__global__ void __launch_bounds__(256) pack_batched_kernel(const ddpm_pack_entry* __restrict__ entries) {
    __shared__ float tile[PK_T][PK_T * 9 + 1];               // +1: the co-fastest read of the dgrad pass is conflict-free
    const ddpm_pack_entry e = entries[blockIdx.y];
    const int taps = e.taps, CiP = e.CiP, CoP = e.CoP, Cin = e.Cin, Cout = e.Cout;
    const float* __restrict__ w = e.w;
    const int tci = (CiP + PK_T - 1) / PK_T, tco = (CoP + PK_T - 1) / PK_T;
    const int row = PK_T * taps;                             // floats per output channel inside a tile
    if (taps > 9) return;                                    // (never: 3x3 and 1x1 only; larger kernels use ddpm_pack_weights)
    for (int t = blockIdx.x; t < tci * tco; t += gridDim.x) {
        const int co0 = (t / tci) * PK_T, ci0 = (t % tci) * PK_T;
        __syncthreads();
        for (int l = threadIdx.x; l < PK_T * row; l += 256) {
            const int r = l / row, k = l - r * row;          // k = ci_local * taps + tap: contiguous in the OIHW source
            const int co = co0 + r, ci = ci0 + k / taps;
            tile[r][k] = (co < Cout && ci < Cin) ? w[((int64_t)co * Cin + ci0) * taps + k] : 0.f;
        }
        __syncthreads();
        for (int l = threadIdx.x; l < PK_T * row; l += 256) {
            // forward copy [co][tap][ci]: ci fastest
            const int c = l % PK_T, rt = l / PK_T, tap = rt % taps, r = rt / taps;
            const int co = co0 + r, ci = ci0 + c;
            if (co < CoP && ci < CiP && e.wf) {
                const float v = tile[r][c * taps + tap];
                const int64_t o = ((int64_t)co * taps + tap) * CiP + ci;
                pack_store(e.wf, e.dtype, o, v);
            }
            // dgrad copy [ci][taps-1-tap][co]: co fastest
            const int r2 = l % PK_T, ct = l / PK_T, tap2 = ct % taps, c2 = ct / taps;
            const int co2 = co0 + r2, ci2 = ci0 + c2;
            if (co2 < CoP && ci2 < CiP && e.wd) {
                const float v = tile[r2][c2 * taps + tap2];
                const int64_t o = ((int64_t)ci2 * taps + (taps - 1 - tap2)) * CoP + co2;
                pack_store(e.wd, e.dtype, o, v);
            }
        }
    }
}
extern "C" int ddpm_pack_weights_batched(const ddpm_pack_entry* entries_dev, int n, void* stream) {
    if (!entries_dev || n <= 0) return DDPM_E_ARG;
    dim3 grid(48, n);
    pack_batched_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(entries_dev);
    LAUNCH_OK();
    return 0;
}
