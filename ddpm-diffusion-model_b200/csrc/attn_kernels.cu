// Spatial self-attention over H*W tokens, reading q/k/v straight out of the NHWC output of the
// 1x1 `qkv` convolution (channel = s*heads*d + head*d + i), so the four permute+contiguous copies
// of attention.py:63-65,72 never exist.  softmax(q k^T / sqrt(d)) v, non-causal (attention.py:69).
//
// Flash-style: K/V tiles staged in shared memory, online softmax, fp32 accumulation.  Attention is
// <0.4 % of model FLOPs (SURVEY.md §5) and N <= 1024 tokens, so this kernel is latency-, not
// tensor-bound; it runs on CUDA cores.
#include "common.cuh"
#include <math.h>

#define AT 128          // threads per block (4 warps)
#define KT 64           // keys per tile
#define QPW 4           // queries per warp
#define DMAX 128

// token p of image n -> (y, x)
template <typename T>
__device__ __forceinline__ const T* tok(const TV& v, int n, int p, int c) { int y = p / v.W; return v.at<T>(n, y, p - y * v.W, c); }
template <typename T>
__device__ __forceinline__ T* tokw(const TV& v, int n, int p, int c) { int y = p / v.W; return v.at<T>(n, y, p - y * v.W, c); }

template <typename T>
__global__ void __launch_bounds__(AT) attn_fwd_kernel(TV qkv, TV out, int heads, int d, float scale, float* lse) {
    extern __shared__ float sm[];
    const int dp = d + 1;
    float* Ks = sm;                       // [KT][dp]
    float* Vs = Ks + KT * dp;             // [KT][dp]
    float* Qs = Vs + KT * dp;             // [4 warps][d]
    float* Ps = Qs + 4 * d;               // [4 warps][KT]
    const int b = blockIdx.z, h = blockIdx.y, N = qkv.H * qkv.W, inner = heads * d;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int qbase = blockIdx.x * (4 * QPW);

    float o[QPW][DMAX / 32], mrun[QPW], lrun[QPW];
#pragma unroll
    for (int qi = 0; qi < QPW; ++qi) {
        mrun[qi] = -INFINITY; lrun[qi] = 0.f;
#pragma unroll
        for (int r = 0; r < DMAX / 32; ++r) o[qi][r] = 0.f;
    }

    for (int k0 = 0; k0 < N; k0 += KT) {
        __syncthreads();
        for (int i = threadIdx.x; i < KT * d; i += AT) {
            int j = i / d, c = i - j * d;
            float kv = 0.f, vv = 0.f;
            if (k0 + j < N) {
                kv = ldf<T>(tok<T>(qkv, b, k0 + j, inner + h * d + c));
                vv = ldf<T>(tok<T>(qkv, b, k0 + j, 2 * inner + h * d + c));
            }
            Ks[j * dp + c] = kv; Vs[j * dp + c] = vv;
        }
        __syncthreads();
#pragma unroll
        for (int qi = 0; qi < QPW; ++qi) {
            const int q = qbase + warp * QPW + qi;
            if (q >= N) break;                                   // warp-uniform
            __syncwarp();
            for (int c = lane; c < d; c += 32) Qs[warp * d + c] = ldf<T>(tok<T>(qkv, b, q, h * d + c)) * scale;
            __syncwarp();
            float s0 = -INFINITY, s1 = -INFINITY;
            if (k0 + lane < N) { float a = 0.f; for (int c = 0; c < d; ++c) a = fmaf(Qs[warp * d + c], Ks[lane * dp + c], a); s0 = a; }
            if (k0 + lane + 32 < N) { float a = 0.f; for (int c = 0; c < d; ++c) a = fmaf(Qs[warp * d + c], Ks[(lane + 32) * dp + c], a); s1 = a; }
            float mt = warp_max(fmaxf(s0, s1));
            float mnew = fmaxf(mrun[qi], mt);
            float corr = __expf(mrun[qi] - mnew);
            float p0 = __expf(s0 - mnew), p1 = __expf(s1 - mnew);
            lrun[qi] = lrun[qi] * corr + warp_sum(p0 + p1);
            mrun[qi] = mnew;
            Ps[warp * KT + lane] = p0; Ps[warp * KT + lane + 32] = p1;
            __syncwarp();
            const int kn = min(KT, N - k0);
            _Pragma("unroll") for (int r = 0; r < DMAX / 32; ++r) {
                int c = lane + 32 * r;
                if (c < d) {
                    float a = o[qi][r] * corr;
                    for (int j = 0; j < kn; ++j) a = fmaf(Ps[warp * KT + j], Vs[j * dp + c], a);
                    o[qi][r] = a;
                }
            }
        }
    }
#pragma unroll
    for (int qi = 0; qi < QPW; ++qi) {
        const int q = qbase + warp * QPW + qi;
        if (q >= N) break;
        float inv = 1.0f / lrun[qi];
        _Pragma("unroll") for (int r = 0; r < DMAX / 32; ++r) {
            int c = lane + 32 * r;
            if (c < d) stf<T>(tokw<T>(out, b, q, h * d + c), o[qi][r] * inv);
        }
        if (lane == 0) lse[((size_t)b * heads + h) * N + q] = mrun[qi] + __logf(lrun[qi]);
    }
}

int attn_tc_supported(const ddpm_tensor* qkv, const ddpm_tensor* out, int heads, int d, int dtype);      // attn_tc.cu
int attn_tc_launch(const ddpm_tensor* qkv, const ddpm_tensor* out, int heads, int d, float* lse, int dtype, cudaStream_t st);
int ddpm_force_simt_flag();
extern "C" int ddpm_attn_fwd(const ddpm_tensor* qkv, const ddpm_tensor* out, int heads, int d, float* lse,
                             int dtype, void* stream) {
    if (!tensor_ok(qkv) || !tensor_ok(out) || !lse || heads <= 0 || d <= 0 || d > DMAX) return DDPM_E_ARG;
    if (qkv->C != 3 * heads * d || out->C != heads * d || out->N != qkv->N || out->H != qkv->H || out->W != qkv->W) return DDPM_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    // tcgen05 forward for bf16 / fp16, head_dim 32 / 64 / 128, W <= 128; everything else on the CUDA cores
    if (!ddpm_force_simt_flag() && attn_tc_supported(qkv, out, heads, d, dtype)) return attn_tc_launch(qkv, out, heads, d, lse, dtype, st);
    int N = qkv->H * qkv->W;
    dim3 grid(ceil_div(N, 4 * QPW), heads, qkv->N);
    size_t smem = sizeof(float) * (2 * KT * (d + 1) + 4 * d + 4 * KT);
    float scale = 1.0f / sqrtf((float)d);
    if (dtype == DDPM_F32) {
        CUDA_TRY(cudaFuncSetAttribute(attn_fwd_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(launch_kernel(attn_fwd_kernel<float>, grid, dim3(AT), smem, st, TV(*qkv), TV(*out), heads, d, scale, lse));
    } else if (dtype == DDPM_BF16) {
        CUDA_TRY(cudaFuncSetAttribute(attn_fwd_kernel<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(launch_kernel(attn_fwd_kernel<bf16>, grid, dim3(AT), smem, st, TV(*qkv), TV(*out), heads, d, scale, lse));
    } else if (dtype == DDPM_F16) {
        CUDA_TRY(cudaFuncSetAttribute(attn_fwd_kernel<f16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(launch_kernel(attn_fwd_kernel<f16>, grid, dim3(AT), smem, st, TV(*qkv), TV(*out), heads, d, scale, lse));
    } else return DDPM_E_ARG;
    LAUNCH_OK();
    return 0;
}

// ------------------------------------------------------------------------------------ backward
// Pass A (per query row): P_ij = exp(scale q_i.k_j - lse_i); dP_ij = dO_i . v_j; D_i = dO_i . O_i;
//   dS_ij = P_ij (dP_ij - D_i); dq_i = scale * sum_j dS_ij k_j.   P and dS go to scratch.
// Pass B (per key row):  dv_j = sum_i P_ij dO_i ; dk_j = scale * sum_i dS_ij q_i.
template <typename T>
__global__ void __launch_bounds__(AT) attn_bwd_q_kernel(TV qkv, TV out, TV dout, TV dqkv, int heads, int d, float scale,
                                                        const float* lse, float* Pm, float* dSm) {
    extern __shared__ float sm[];
    const int dp = d + 1;
    float* Ks = sm; float* Vs = Ks + KT * dp;
    float* Qs = Vs + KT * dp;             // [4][d]   q * scale
    float* Gs = Qs + 4 * d;               // [4][d]   dO
    float* Ss = Gs + 4 * d;               // [4][KT]  dS of the tile
    const int b = blockIdx.z, h = blockIdx.y, N = qkv.H * qkv.W, inner = heads * d;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int qbase = blockIdx.x * (4 * QPW);
    const size_t mat = ((size_t)b * heads + h) * N * N;

    float dq[QPW][DMAX / 32], Di[QPW], Li[QPW];
#pragma unroll
    for (int qi = 0; qi < QPW; ++qi) {
        const int q = qbase + warp * QPW + qi;
        Di[qi] = 0.f; Li[qi] = 0.f;
#pragma unroll
        for (int r = 0; r < DMAX / 32; ++r) dq[qi][r] = 0.f;
        if (q < N) {
            float a = 0.f;
            for (int c = lane; c < d; c += 32)
                a = fmaf(ldf<T>(tok<T>(dout, b, q, h * d + c)), ldf<T>(tok<T>(out, b, q, h * d + c)), a);
            Di[qi] = warp_sum(a);
            Li[qi] = lse[((size_t)b * heads + h) * N + q];
        }
    }
    for (int k0 = 0; k0 < N; k0 += KT) {
        __syncthreads();
        for (int i = threadIdx.x; i < KT * d; i += AT) {
            int j = i / d, c = i - j * d;
            float kv = 0.f, vv = 0.f;
            if (k0 + j < N) {
                kv = ldf<T>(tok<T>(qkv, b, k0 + j, inner + h * d + c));
                vv = ldf<T>(tok<T>(qkv, b, k0 + j, 2 * inner + h * d + c));
            }
            Ks[j * dp + c] = kv; Vs[j * dp + c] = vv;
        }
        __syncthreads();
#pragma unroll
        for (int qi = 0; qi < QPW; ++qi) {
            const int q = qbase + warp * QPW + qi;
            if (q >= N) break;
            __syncwarp();
            for (int c = lane; c < d; c += 32) {
                Qs[warp * d + c] = ldf<T>(tok<T>(qkv, b, q, h * d + c)) * scale;
                Gs[warp * d + c] = ldf<T>(tok<T>(dout, b, q, h * d + c));
            }
            __syncwarp();
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                int j = lane + 32 * half;
                float ds = 0.f;
                if (k0 + j < N) {
                    float s = 0.f, dpv = 0.f;
                    for (int c = 0; c < d; ++c) {
                        s = fmaf(Qs[warp * d + c], Ks[j * dp + c], s);
                        dpv = fmaf(Gs[warp * d + c], Vs[j * dp + c], dpv);
                    }
                    float pij = __expf(s - Li[qi]);
                    ds = pij * (dpv - Di[qi]);
                    Pm[mat + (size_t)q * N + k0 + j] = pij;
                    dSm[mat + (size_t)q * N + k0 + j] = ds;
                }
                Ss[warp * KT + j] = ds;
            }
            __syncwarp();
            const int kn = min(KT, N - k0);
            _Pragma("unroll") for (int r = 0; r < DMAX / 32; ++r) {
                int c = lane + 32 * r;
                if (c < d) {
                    float a = dq[qi][r];
                    for (int j = 0; j < kn; ++j) a = fmaf(Ss[warp * KT + j], Ks[j * dp + c], a);
                    dq[qi][r] = a;
                }
            }
        }
    }
#pragma unroll
    for (int qi = 0; qi < QPW; ++qi) {
        const int q = qbase + warp * QPW + qi;
        if (q >= N) break;
        _Pragma("unroll") for (int r = 0; r < DMAX / 32; ++r) {
            int c = lane + 32 * r;
            if (c < d) stf<T>(tokw<T>(dqkv, b, q, h * d + c), dq[qi][r] * scale);
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(AT) attn_bwd_kv_kernel(TV qkv, TV dout, TV dqkv, int heads, int d, float scale,
                                                         const float* Pm, const float* dSm) {
    extern __shared__ float sm[];
    const int dp = d + 1;
    float* Qt = sm;                       // [KT queries][dp]
    float* Gt = Qt + KT * dp;             // [KT queries][dp]  dO
    float* Pt = Gt + KT * dp;             // [KT queries][16 keys + 1]
    float* St = Pt + KT * 17;             // [KT queries][16 keys + 1]
    const int b = blockIdx.z, h = blockIdx.y, N = qkv.H * qkv.W, inner = heads * d;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int jbase = blockIdx.x * 16;    // 16 keys per block, 4 per warp
    const size_t mat = ((size_t)b * heads + h) * N * N;
    float dk[4][DMAX / 32], dv[4][DMAX / 32];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int r = 0; r < DMAX / 32; ++r) { dk[a][r] = 0.f; dv[a][r] = 0.f; }

    for (int i0 = 0; i0 < N; i0 += KT) {
        __syncthreads();
        for (int i = threadIdx.x; i < KT * d; i += AT) {
            int qi = i / d, c = i - qi * d;
            float qv = 0.f, gv = 0.f;
            if (i0 + qi < N) {
                qv = ldf<T>(tok<T>(qkv, b, i0 + qi, h * d + c));
                gv = ldf<T>(tok<T>(dout, b, i0 + qi, h * d + c));
            }
            Qt[qi * dp + c] = qv; Gt[qi * dp + c] = gv;
        }
        for (int i = threadIdx.x; i < KT * 16; i += AT) {
            int qi = i >> 4, jj = i & 15;
            float pv = 0.f, sv = 0.f;
            if (i0 + qi < N && jbase + jj < N) {
                pv = Pm[mat + (size_t)(i0 + qi) * N + jbase + jj];
                sv = dSm[mat + (size_t)(i0 + qi) * N + jbase + jj];
            }
            Pt[qi * 17 + jj] = pv; St[qi * 17 + jj] = sv;
        }
        __syncthreads();
        const int qn = min(KT, N - i0);
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            int jj = warp * 4 + a;
            _Pragma("unroll") for (int r = 0; r < DMAX / 32; ++r) {
                int c = lane + 32 * r;
                if (c < d) {
                    float ak = dk[a][r], av = dv[a][r];
                    for (int qi = 0; qi < qn; ++qi) {
                        ak = fmaf(St[qi * 17 + jj], Qt[qi * dp + c], ak);
                        av = fmaf(Pt[qi * 17 + jj], Gt[qi * dp + c], av);
                    }
                    dk[a][r] = ak; dv[a][r] = av;
                }
            }
        }
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        int j = jbase + warp * 4 + a;
        if (j >= N) break;
        _Pragma("unroll") for (int r = 0; r < DMAX / 32; ++r) {
            int c = lane + 32 * r;
            if (c < d) {
                stf<T>(tokw<T>(dqkv, b, j, inner + h * d + c), dk[a][r] * scale);
                stf<T>(tokw<T>(dqkv, b, j, 2 * inner + h * d + c), dv[a][r]);
            }
        }
    }
}

int64_t attn_tc_bwd_scratch_floats(const ddpm_tensor* qkv, const ddpm_tensor* out, int heads, int d, int dtype);      // attn_tc.cu
int attn_tc_bwd_launch(const ddpm_tensor* qkv, const ddpm_tensor* out, const ddpm_tensor* dout, const float* lse,
                       const ddpm_tensor* dqkv, int heads, int d, float* scratch, int dtype, cudaStream_t st);
extern "C" int64_t ddpm_attn_bwd_scratch_floats(const ddpm_tensor* qkv, const ddpm_tensor* out, int heads, int d, int dtype) {
    if (!tensor_ok(qkv) || !tensor_ok(out) || heads <= 0 || d <= 0) return 0;
    const int64_t N = (int64_t)qkv->H * qkv->W;
    if (!ddpm_force_simt_flag()) {
        const int64_t tc = attn_tc_bwd_scratch_floats(qkv, out, heads, d, dtype);
        if (tc > 0) return tc;                             // tensor-core backward: D = dO . O per query only
    }
    return 2 * (int64_t)qkv->N * heads * N * N;             // CUDA-core backward: P and dS
}
extern "C" int ddpm_attn_bwd(const ddpm_tensor* qkv, const ddpm_tensor* out, const ddpm_tensor* dout,
                             const float* lse, const ddpm_tensor* dqkv, int heads, int d, float* scratch,
                             int dtype, void* stream) {
    if (!tensor_ok(qkv) || !tensor_ok(out) || !tensor_ok(dout) || !tensor_ok(dqkv) || !lse || !scratch) return DDPM_E_ARG;
    if (heads <= 0 || d <= 0 || d > DMAX || qkv->C != 3 * heads * d || dqkv->C != qkv->C || out->C != heads * d || dout->C != out->C) return DDPM_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    // tcgen05 backward with P recomputed from lse (no N x N scratch) whenever qkv / out are eligible; CUDA cores otherwise.
    // ddpm_attn_bwd_scratch_floats sizes the scratch from qkv / out alone, so dout / dqkv that the tensor-core kernels cannot
    // take are rejected rather than sent to the CUDA-core kernels, which would write N x N matrices into that scratch.
    if (!ddpm_force_simt_flag() && attn_tc_supported(qkv, out, heads, d, dtype)) {
        if (!attn_tc_supported(dqkv, dout, heads, d, dtype) || dout->halo != qkv->halo) return DDPM_E_ARG;
        const ddpm_tensor* same[3] = {out, dout, dqkv};
        for (const ddpm_tensor* t : same)
            if (t->N != qkv->N || t->H != qkv->H || t->W != qkv->W) return DDPM_E_ARG;
        return attn_tc_bwd_launch(qkv, out, dout, lse, dqkv, heads, d, scratch, dtype, st);
    }
    int N = qkv->H * qkv->W;
    float* Pm = scratch; float* dSm = scratch + (size_t)qkv->N * heads * N * N;
    float scale = 1.0f / sqrtf((float)d);
    dim3 gq(ceil_div(N, 4 * QPW), heads, qkv->N), gk(ceil_div(N, 16), heads, qkv->N);
    size_t smq = sizeof(float) * (2 * KT * (d + 1) + 8 * d + 4 * KT);
    size_t smk = sizeof(float) * (2 * KT * (d + 1) + 2 * KT * 17);
#define GO(T) { \
        CUDA_TRY(cudaFuncSetAttribute(attn_bwd_q_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smq)); \
        CUDA_TRY(cudaFuncSetAttribute(attn_bwd_kv_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smk)); \
        CUDA_TRY(launch_kernel(attn_bwd_q_kernel<T>, gq, dim3(AT), smq, st, TV(*qkv), TV(*out), TV(*dout), TV(*dqkv), heads, d, scale, (const float*)lse, Pm, dSm)); \
        LAUNCH_OK(); \
        CUDA_TRY(launch_kernel(attn_bwd_kv_kernel<T>, gk, dim3(AT), smk, st, TV(*qkv), TV(*dout), TV(*dqkv), heads, d, scale, (const float*)Pm, (const float*)dSm)); \
        LAUNCH_OK(); }
    if (dtype == DDPM_F32) GO(float) else if (dtype == DDPM_BF16) GO(bf16) else if (dtype == DDPM_F16) GO(f16) else return DDPM_E_ARG;
#undef GO
    return 0;
}
