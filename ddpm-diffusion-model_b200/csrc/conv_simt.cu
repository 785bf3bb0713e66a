// Generic implicit-GEMM convolution / linear on CUDA cores (fp32 accumulate).
//
// This is the *exact-arithmetic* path: fp32 activations for the 1e-4 parity target, and every shape
// the tcgen05 kernel (conv_tc.cu) does not take (K=27 in_conv, N=3 out_conv, stride-2 and
// transposed gathers, tiny linears).  ddpm_conv / ddpm_conv_wgrad in abi_conv.cu dispatch.
//
// fprop  : out[n,oy,ox,co] = epi( sum_{ky,kx,ci} A(n, oy*s+ky-p, ox*s+kx-p, ci) * W[co][ky][kx][ci] )
// dgrad  : same kernel on dY with flipped/transposed weights; stride-2 uses the TRANSPOSED gather
// wgrad  : dW[co][ci][ky][kx] += sum_{n,oy,ox} dY[n,oy,ox,co] * A(n, oy*s+ky-p, ox*s+kx-p, ci)
//
// Replaces cuDNN/cuBLAS calls behind nn.Conv2d / nn.Linear (unet_backbone.py:22,27,32,35,51,60,97,100;
// attention.py:30,32,53-54).
#include "common.cuh"

#define BM 64
#define BN 64
#define BK 16
#define CT 256

struct ConvP {
    TV in, out, res, z;
    const void* w; const float* bias; const float* tbias; int tbias_pitch;
    int KH, KW, stride, pad, mode, a_silu, epi;
    int Cin, Cout, M, Kt, HoWo, bias_n;
    int vecA, vecB, vecO, has_res, has_z;
};

template <typename T>
__global__ void __launch_bounds__(CT) conv_simt_kernel(ConvP p) {
    __shared__ float As[BK][BM + 4];
    __shared__ float Bs[BK][BN + 4];
    const int tid = threadIdx.x;
    const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
    const T* __restrict__ w = reinterpret_cast<const T*>(p.w);

    // A-load role: row ar (0..63), k quad akq
    const int ar = tid >> 2, akq = (tid & 3) * 4;
    const int am = m0 + ar;
    int an = 0, aoy = 0, aox = 0; bool arow_ok = am < p.M;
    if (arow_ok) { an = am / p.HoWo; int r = am - an * p.HoWo; aoy = r / p.out.W; aox = r - aoy * p.out.W; }
    // B-load role: col bc (0..63), k quad akq
    const int bc = tid >> 2;
    const bool bcol_ok = (n0 + bc) < p.Cout;
    const T* wrow = w + (int64_t)(n0 + bc) * p.Kt;

    const int ty = tid >> 4, tx = tid & 15;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    for (int k0 = 0; k0 < p.Kt; k0 += BK) {
        // ---- gather A
        float av[4] = {0.f, 0.f, 0.f, 0.f};
        {
            const int k = k0 + akq;
            if (arow_ok && k < p.Kt) {
                if (p.vecA) {
                    int tap = k / p.Cin, ci = k - tap * p.Cin;
                    int ky = tap / p.KW, kx = tap - ky * p.KW;
                    int iy, ix; bool ok;
                    if (p.mode == DDPM_CONV_NORMAL) {
                        iy = aoy * p.stride + ky - p.pad; ix = aox * p.stride + kx - p.pad;
                        ok = iy >= 0 && iy < p.in.H && ix >= 0 && ix < p.in.W;
                    } else {
                        int u = aoy + ky - p.pad, v = aox + kx - p.pad;
                        ok = u >= 0 && v >= 0 && (u % p.stride) == 0 && (v % p.stride) == 0;
                        iy = u / p.stride; ix = v / p.stride;
                        ok = ok && iy < p.in.H && ix < p.in.W;
                    }
                    if (ok) {
                        const T* src = p.in.at<T>(an, iy, ix, ci);
                        if (sizeof(T) == 4) {
                            float4 t = *reinterpret_cast<const float4*>(src);
                            av[0] = t.x; av[1] = t.y; av[2] = t.z; av[3] = t.w;
                        } else {
                            uint2 t = *reinterpret_cast<const uint2*>(src);
                            float2 a = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&t.x));
                            float2 b = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&t.y));
                            av[0] = a.x; av[1] = a.y; av[2] = b.x; av[3] = b.y;
                        }
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        int kk = k + j;
                        if (kk < p.Kt) {
                            int tap = kk / p.Cin, ci = kk - tap * p.Cin;
                            int ky = tap / p.KW, kx = tap - ky * p.KW;
                            int iy, ix; bool ok;
                            if (p.mode == DDPM_CONV_NORMAL) {
                                iy = aoy * p.stride + ky - p.pad; ix = aox * p.stride + kx - p.pad;
                                ok = iy >= 0 && iy < p.in.H && ix >= 0 && ix < p.in.W;
                            } else {
                                int u = aoy + ky - p.pad, v = aox + kx - p.pad;
                                ok = u >= 0 && v >= 0 && (u % p.stride) == 0 && (v % p.stride) == 0;
                                iy = u / p.stride; ix = v / p.stride;
                                ok = ok && iy < p.in.H && ix < p.in.W;
                            }
                            if (ok) av[j] = ldf<T>(p.in.at<T>(an, iy, ix, ci));
                        }
                    }
                }
                if (p.a_silu) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) av[j] = silu_f(av[j]);
                }
            }
        }
        // ---- load B
        float bv[4] = {0.f, 0.f, 0.f, 0.f};
        {
            const int k = k0 + akq;
            if (bcol_ok && k < p.Kt) {
                if (p.vecB) {
                    if (sizeof(T) == 4) {
                        float4 t = *reinterpret_cast<const float4*>(wrow + k);
                        bv[0] = t.x; bv[1] = t.y; bv[2] = t.z; bv[3] = t.w;
                    } else {
                        uint2 t = *reinterpret_cast<const uint2*>(wrow + k);
                        float2 a = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&t.x));
                        float2 b = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&t.y));
                        bv[0] = a.x; bv[1] = a.y; bv[2] = b.x; bv[3] = b.y;
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j) if (k + j < p.Kt) bv[j] = ldf<T>(wrow + k + j);
                }
            }
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 4; ++j) { As[akq + j][ar] = av[j]; Bs[akq + j][bc] = bv[j]; }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            float aa[4] = {a.x, a.y, a.z, a.w}, bb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(aa[i], bb[j], acc[i][j]);
        }
    }

    // ---- epilogue
    const float* tb = p.tbias;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int m = m0 + ty * 4 + i;
        if (m >= p.M) continue;
        int n = m / p.HoWo; int r = m - n * p.HoWo; int oy = r / p.out.W, ox = r - oy * p.out.W;
        int co0 = n0 + tx * 4;
        if (co0 >= p.Cout) continue;
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int co = co0 + j;
            float x = acc[i][j];
            if (co < p.Cout) {
                if (p.bias && co < p.bias_n) x += p.bias[co];
                if (tb) x += tb[(int64_t)n * p.tbias_pitch + co];
                if (p.has_res) x += ldf<T>(p.res.at<T>(n, oy, ox, co));
                if (p.has_z) x *= dsilu_f(ldf<T>(p.z.at<T>(n, oy, ox, co)));
                if (p.epi & DDPM_EPI_ACCUM) x += ldf<T>(p.out.at<T>(n, oy, ox, co));
            }
            v[j] = x;
        }
        T* dst = p.out.at<T>(n, oy, ox, co0);
        if (p.vecO && co0 + 3 < p.Cout) {
            if (sizeof(T) == 4) *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
            else {
                uint2 t;
                *reinterpret_cast<__nv_bfloat162*>(&t.x) = __floats2bfloat162_rn(v[0], v[1]);
                *reinterpret_cast<__nv_bfloat162*>(&t.y) = __floats2bfloat162_rn(v[2], v[3]);
                *reinterpret_cast<uint2*>(dst) = t;
            }
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) if (co0 + j < p.Cout) stf<T>(dst + j, v[j]);
        }
    }
}

static inline bool al(const void* p, int bytes) { return (((uintptr_t)p) % bytes) == 0; }

// ------------------------------------------------------------------------------------ small linear
// nn.Linear on the fp32 time path (attention.py:30,32; unet_backbone.py:27): out[b][n] = sum_k f(x[b][k]) W[n][k]
// (+ bias, * silu'(z), += out).  M = batch, N, K <= a few hundred: the generic 64x64 tile above runs them on
// 6 CTAs with an unpipelined 32-trip K loop (42 us each, 31 launches per step).  Here: 32x32 tiles (4x the CTAs),
// BK = 32, register prefetch + double-buffered shared memory (one barrier per trip).
#define LBM 32
#define LBN 32
#define LBK 32
struct LinP {
    const float* x; const float* w; const float* bias; const float* z; float* out;
    int M, N, K, xpitch, opitch, zpitch, a_silu, accum, bias_n, vec;
};
__global__ void __launch_bounds__(256) linear_small_kernel(LinP p) {
    __shared__ float As[2][LBK][LBM + 1];
    __shared__ float Bs[2][LBK][LBN + 1];
    const int tid = threadIdx.x;
    const int m0 = blockIdx.x * LBM, n0 = blockIdx.y * LBN;
    const int lr = tid >> 3, kq = (tid & 7) * 4;
    const int ty = tid >> 4, tx = tid & 15;
    const bool aok = (m0 + lr) < p.M, bok = (n0 + lr) < p.N;
    const float* xrow = p.x + (int64_t)(m0 + lr) * p.xpitch;
    const float* wrow = p.w + (int64_t)(n0 + lr) * p.K;
    float av[4], bv[4];
    auto fetch = [&](int k0) {
#pragma unroll
        for (int j = 0; j < 4; ++j) { av[j] = 0.f; bv[j] = 0.f; }
        const int k = k0 + kq;
        if (p.vec && k + 3 < p.K) {
            if (aok) { float4 t = *reinterpret_cast<const float4*>(xrow + k); av[0] = t.x; av[1] = t.y; av[2] = t.z; av[3] = t.w; }
            if (bok) { float4 t = __ldg(reinterpret_cast<const float4*>(wrow + k)); bv[0] = t.x; bv[1] = t.y; bv[2] = t.z; bv[3] = t.w; }
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) if (k + j < p.K) { if (aok) av[j] = xrow[k + j]; if (bok) bv[j] = __ldg(wrow + k + j); }
        }
        if (p.a_silu) {
#pragma unroll
            for (int j = 0; j < 4; ++j) av[j] = silu_f(av[j]);
        }
    };
    float acc[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
    fetch(0);
    int buf = 0;
    for (int k0 = 0; k0 < p.K; k0 += LBK, buf ^= 1) {
#pragma unroll
        for (int j = 0; j < 4; ++j) { As[buf][kq + j][lr] = av[j]; Bs[buf][kq + j][lr] = bv[j]; }
        __syncthreads();
        if (k0 + LBK < p.K) fetch(k0 + LBK);                 // next trip's loads are in flight during the FMAs
#pragma unroll
        for (int kk = 0; kk < LBK; ++kk) {
            const float a0 = As[buf][kk][ty * 2], a1 = As[buf][kk][ty * 2 + 1];
            const float b0 = Bs[buf][kk][tx * 2], b1 = Bs[buf][kk][tx * 2 + 1];
            acc[0][0] = fmaf(a0, b0, acc[0][0]); acc[0][1] = fmaf(a0, b1, acc[0][1]);
            acc[1][0] = fmaf(a1, b0, acc[1][0]); acc[1][1] = fmaf(a1, b1, acc[1][1]);
        }
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const int m = m0 + ty * 2 + i;
        if (m >= p.M) continue;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int n = n0 + tx * 2 + j;
            if (n >= p.N) continue;
            float v = acc[i][j];
            if (p.bias && n < p.bias_n) v += p.bias[n];
            if (p.z) v *= dsilu_f(p.z[(int64_t)m * p.zpitch + n]);
            float* o = p.out + (int64_t)m * p.opitch + n;
            if (p.accum) v += *o;
            *o = v;
        }
    }
}

static bool linear_small_ok(const ddpm_conv_args* a) {
    return a->dtype == DDPM_F32 && a->KH == 1 && a->KW == 1 && a->stride == 1 && a->pad == 0 && a->mode == DDPM_CONV_NORMAL &&
           a->in.H == 1 && a->in.W == 1 && a->in.halo == 0 && a->out.halo == 0 && !a->res.ptr && !a->tbias &&
           (!a->z.ptr || (a->z.H == 1 && a->z.W == 1 && a->z.halo == 0));
}
static int linear_small_launch(const ddpm_conv_args* a, cudaStream_t st) {
    LinP p;
    p.x = (const float*)a->in.ptr; p.w = (const float*)a->w; p.bias = a->bias; p.z = (const float*)a->z.ptr; p.out = (float*)a->out.ptr;
    p.M = a->in.N; p.N = a->out.C; p.K = a->in.C; p.xpitch = a->in.pitch; p.opitch = a->out.pitch; p.zpitch = a->z.ptr ? a->z.pitch : 0;
    p.a_silu = a->a_silu; p.accum = (a->epi & DDPM_EPI_ACCUM) ? 1 : 0; p.bias_n = a->bias_n > 0 ? a->bias_n : a->out.C;
    p.vec = (p.K % 4 == 0) && (p.xpitch % 4 == 0) && al(p.x, 16) && al(p.w, 16);
    dim3 grid(ceil_div(p.M, LBM), ceil_div(p.N, LBN));
    CUDA_TRY(launch_kernel(linear_small_kernel, grid, dim3(256), 0, st, p));
    LAUNCH_OK();
    return 0;
}

// ------------------------------------------------------------------------------------ time path, batched
// All `time_proj` linears of the UNet (unet_backbone.py:27; 14 / 27 of them, same input silu(temb)) in ONE launch,
// and the whole backward of one of them (dW, db and the accumulated d temb) in ONE launch instead of three.
// 32x32 output tiles, inner tiles of 32, operands fetched through small functors so the same tile routine serves
// row-major and transposed accesses.
// KA / KB: the operand is contiguous along the INNER dimension in global memory -> consecutive threads fetch consecutive
// inner indices (coalesced) and the 33-float row padding makes the transposing shared-memory write conflict-free; otherwise
// consecutive threads fetch consecutive rows.  (Row-fastest fetches of a k-contiguous operand were 1024 strided 4-byte
// loads per tile: the grouped time-proj forward took 80 us for 0.26 GFLOP.)
template <bool KA, bool KB, typename FA, typename FB>
__device__ __forceinline__ void tile_gemm32(FA fa, FB fb, int Kin, float acc[2][2], float (*As)[LBM + 1], float (*Bs)[LBN + 1]) {
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    for (int k0 = 0; k0 < Kin; k0 += LBK) {
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 4; ++j) {                       // 1024 elements per operand tile, 256 threads
            const int l = tid + j * 256;
            if (KA) As[l & 31][l >> 5] = fa(l >> 5, k0 + (l & 31));
            else As[l >> 5][l & 31] = fa(l & 31, k0 + (l >> 5));
            if (KB) Bs[l & 31][l >> 5] = fb(l >> 5, k0 + (l & 31));
            else Bs[l >> 5][l & 31] = fb(l & 31, k0 + (l >> 5));
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < LBK; ++kk) {
            const float a0 = As[kk][ty * 2], a1 = As[kk][ty * 2 + 1];
            const float b0 = Bs[kk][tx * 2], b1 = Bs[kk][tx * 2 + 1];
            acc[0][0] = fmaf(a0, b0, acc[0][0]); acc[0][1] = fmaf(a0, b1, acc[0][1]);
            acc[1][0] = fmaf(a1, b0, acc[1][0]); acc[1][1] = fmaf(a1, b1, acc[1][1]);
        }
    }
}

__global__ void __launch_bounds__(256) linear_grouped_fwd_kernel(const float* __restrict__ x, int M, int K, int xpitch,
                                                                 const ddpm_lin_entry* __restrict__ entries, float* out, int opitch, int a_silu) {
    __shared__ float As[LBK][LBM + 1];
    __shared__ float Bs[LBK][LBN + 1];
    const ddpm_lin_entry e = entries[blockIdx.z];
    const int m0 = blockIdx.x * LBM, n0 = blockIdx.y * LBN;
    if (n0 >= e.N) return;
    const float* __restrict__ w = e.w;
    float acc[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
    tile_gemm32<true, true>([&](int r, int k) { const int m = m0 + r; float v = (m < M && k < K) ? x[(int64_t)m * xpitch + k] : 0.f; return a_silu ? silu_f(v) : v; },
                [&](int r, int k) { const int n = n0 + r; return (n < e.N && k < K) ? __ldg(w + (int64_t)n * K + k) : 0.f; },
                K, acc, As, Bs);
    const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int m = m0 + ty * 2 + i, n = n0 + tx * 2 + j;
            if (m < M && n < e.N) out[(int64_t)m * opitch + e.col0 + n] = acc[i][j] + (e.bias ? e.bias[n] : 0.f) + (e.bias2 ? e.bias2[n] : 0.f);
        }
}

extern "C" int ddpm_linear_grouped_fwd(const float* x, int M, int K, int xpitch, const ddpm_lin_entry* entries_dev, int n,
                                       int max_N, float* out, int out_pitch, int a_silu, void* stream) {
    if (!x || !entries_dev || !out || M <= 0 || K <= 0 || n <= 0 || max_N <= 0) return DDPM_E_ARG;
    dim3 grid(ceil_div(M, LBM), ceil_div(max_N, LBN), n);
    CUDA_TRY(launch_kernel(linear_grouped_fwd_kernel, grid, dim3(256), 0, (cudaStream_t)stream, x, M, K, xpitch, entries_dev, out, out_pitch, a_silu));
    LAUNCH_OK();
    return 0;
}

// y = W silu(temb) + b for one block.  Given dy = dtb [B][N]:  dW[n][k] += sum_b dy[b][n] silu(temb[b][k]),
// db[n] += sum_b dy[b][n],  dtemb[b][k] (+)= (sum_n dy[b][n] W[n][k]) * silu'(temb[b][k]).
__global__ void __launch_bounds__(256) time_proj_bwd_kernel(const float* __restrict__ temb, int B, int K, const float* __restrict__ dy,
                                                            int dpitch, int N, const float* __restrict__ w, float* dw, float* db,
                                                            float* dtemb, int accum, int tilesA_n) {
    __shared__ float As[LBK][LBM + 1];
    __shared__ float Bs[LBK][LBN + 1];
    const int kt = blockIdx.x, r = blockIdx.y;               // K tile; row tile of part A (n) or part B (b)
    const int k0 = kt * LBN;
    const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
    float acc[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
    if (r < tilesA_n) {                                      // ---- part A: weight (and bias) gradient, inner dim = batch
        const int n0 = r * LBM;
        tile_gemm32<false, false>([&](int rr, int b) { const int n = n0 + rr; return (n < N && b < B) ? dy[(int64_t)b * dpitch + n] : 0.f; },
                    [&](int rr, int b) { const int k = k0 + rr; return (k < K && b < B) ? silu_f(temb[(int64_t)b * K + k]) : 0.f; },
                    B, acc, As, Bs);
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int n = n0 + ty * 2 + i, k = k0 + tx * 2 + j;
                if (n < N && k < K) dw[(int64_t)n * K + k] += acc[i][j];
            }
        if (kt == 0 && db && threadIdx.x < LBM) {
            const int n = n0 + threadIdx.x;
            if (n < N) { float s = 0.f; for (int b = 0; b < B; ++b) s += dy[(int64_t)b * dpitch + n]; db[n] += s; }
        }
    } else {                                                 // ---- part B: d temb, inner dim = N
        const int b0 = (r - tilesA_n) * LBM;
        tile_gemm32<true, false>([&](int rr, int n) { const int b = b0 + rr; return (b < B && n < N) ? dy[(int64_t)b * dpitch + n] : 0.f; },
                    [&](int rr, int n) { const int k = k0 + rr; return (k < K && n < N) ? __ldg(w + (int64_t)n * K + k) : 0.f; },
                    N, acc, As, Bs);
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int b = b0 + ty * 2 + i, k = k0 + tx * 2 + j;
                if (b < B && k < K) {
                    const float v = acc[i][j] * dsilu_f(temb[(int64_t)b * K + k]);
                    float* o = dtemb + (int64_t)b * K + k;
                    *o = accum ? *o + v : v;
                }
            }
    }
}

extern "C" int ddpm_time_proj_bwd(const float* temb, int B, int K, const float* dy, int dy_pitch, int N, const float* w,
                                  float* dw, float* db, float* dtemb, int accum_dtemb, void* stream) {
    if (!temb || !dy || !w || !dw || !dtemb || B <= 0 || K <= 0 || N <= 0) return DDPM_E_ARG;
    const int tilesA = ceil_div(N, LBM), tilesB = ceil_div(B, LBM);
    dim3 grid(ceil_div(K, LBN), tilesA + tilesB);
    CUDA_TRY(launch_kernel(time_proj_bwd_kernel, grid, dim3(256), 0, (cudaStream_t)stream, temb, B, K, dy, dy_pitch, N, w, dw, db, dtemb, accum_dtemb, tilesA));
    LAUNCH_OK();
    return 0;
}

int conv_simt_launch(const ddpm_conv_args* a, cudaStream_t st) {
    if (linear_small_ok(a)) return linear_small_launch(a, st);
    ConvP p;
    p.in = TV(a->in); p.out = TV(a->out);
    p.has_res = a->res.ptr != nullptr; p.has_z = a->z.ptr != nullptr;
    p.res = p.has_res ? TV(a->res) : TV(a->out);
    p.z = p.has_z ? TV(a->z) : TV(a->out);
    p.w = a->w; p.bias = a->bias; p.tbias = a->tbias; p.tbias_pitch = a->tbias_pitch;
    p.KH = a->KH; p.KW = a->KW; p.stride = a->stride; p.pad = a->pad; p.mode = a->mode;
    p.a_silu = a->a_silu; p.epi = a->epi;
    p.Cin = a->in.C; p.Cout = a->out.C; p.bias_n = a->bias_n > 0 ? a->bias_n : a->out.C;
    p.HoWo = a->out.H * a->out.W; p.M = a->out.N * p.HoWo; p.Kt = a->KH * a->KW * p.Cin;
    const int es = a->dtype == DDPM_F32 ? 4 : 2;
    p.vecA = (p.Cin % 4 == 0) && (a->in.pitch % 4 == 0) && al(a->in.ptr, 4 * es);
    p.vecB = (p.Kt % 4 == 0) && al(a->w, 4 * es);
    p.vecO = (a->out.pitch % 4 == 0) && al(a->out.ptr, 4 * es);
    dim3 grid(ceil_div(p.M, BM), ceil_div(p.Cout, BN));
    if (a->dtype == DDPM_F32) CUDA_TRY(launch_kernel(conv_simt_kernel<float>, grid, dim3(CT), 0, st, p));
    else CUDA_TRY(launch_kernel(conv_simt_kernel<bf16>, grid, dim3(CT), 0, st, p));
    LAUNCH_OK();
    return 0;
}

// ------------------------------------------------------------------------------------ wgrad
struct WgP {
    TV act, dy;
    float* dw;
    int KH, KW, stride, pad, a_silu;
    int Cin, Cout, Q, Kf, HoWo, qper, CinV, CoutV;
    int vecA, vecY;
};

template <typename T>
__global__ void __launch_bounds__(CT) wgrad_simt_kernel(WgP p) {
    __shared__ float Ys[BK][BM + 4];   // [q][co]
    __shared__ float Xs[BK][BN + 4];   // [q][kf]
    const int tid = threadIdx.x;
    const int co0 = blockIdx.x * BM, kf0 = blockIdx.y * BN;
    const int qbeg = blockIdx.z * p.qper, qend = min(p.Q, qbeg + p.qper);
    const int lq = tid >> 4, l4 = (tid & 15) * 4;
    const int ty = tid >> 4, tx = tid & 15;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    // this thread's 4 kf columns (fixed across the loop)
    int tap[4], ci[4]; bool kok[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        int kf = kf0 + l4 + j; kok[j] = kf < p.Kf;
        tap[j] = kok[j] ? kf / p.Cin : 0; ci[j] = kok[j] ? kf - tap[j] * p.Cin : 0;
    }

    for (int q0 = qbeg; q0 < qend; q0 += BK) {
        const int q = q0 + lq;
        float yv[4] = {0.f, 0.f, 0.f, 0.f}, xv[4] = {0.f, 0.f, 0.f, 0.f};
        if (q < qend) {
            int n = q / p.HoWo; int r = q - n * p.HoWo; int oy = r / p.dy.W, ox = r - oy * p.dy.W;
            // dY[q][co0+l4 .. +3]
            if (co0 + l4 < p.Cout) {
                const T* src = p.dy.at<T>(n, oy, ox, co0 + l4);
                if (p.vecY && co0 + l4 + 3 < p.Cout) {
                    if (sizeof(T) == 4) { float4 t = *reinterpret_cast<const float4*>(src); yv[0] = t.x; yv[1] = t.y; yv[2] = t.z; yv[3] = t.w; }
                    else {
                        uint2 t = *reinterpret_cast<const uint2*>(src);
                        float2 a = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&t.x));
                        float2 b = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&t.y));
                        yv[0] = a.x; yv[1] = a.y; yv[2] = b.x; yv[3] = b.y;
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j) if (co0 + l4 + j < p.Cout) yv[j] = ldf<T>(src + j);
                }
            }
            // A[q][kf0+l4 .. +3]
            if (p.vecA && kok[3]) {
                int ky = tap[0] / p.KW, kx = tap[0] - ky * p.KW;
                int iy = oy * p.stride + ky - p.pad, ix = ox * p.stride + kx - p.pad;
                if (iy >= 0 && iy < p.act.H && ix >= 0 && ix < p.act.W) {
                    const T* src = p.act.at<T>(n, iy, ix, ci[0]);
                    if (sizeof(T) == 4) { float4 t = *reinterpret_cast<const float4*>(src); xv[0] = t.x; xv[1] = t.y; xv[2] = t.z; xv[3] = t.w; }
                    else {
                        uint2 t = *reinterpret_cast<const uint2*>(src);
                        float2 a = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&t.x));
                        float2 b = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&t.y));
                        xv[0] = a.x; xv[1] = a.y; xv[2] = b.x; xv[3] = b.y;
                    }
                }
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (!kok[j]) continue;
                    int ky = tap[j] / p.KW, kx = tap[j] - ky * p.KW;
                    int iy = oy * p.stride + ky - p.pad, ix = ox * p.stride + kx - p.pad;
                    if (iy >= 0 && iy < p.act.H && ix >= 0 && ix < p.act.W) xv[j] = ldf<T>(p.act.at<T>(n, iy, ix, ci[j]));
                }
            }
            if (p.a_silu) {
#pragma unroll
                for (int j = 0; j < 4; ++j) xv[j] = kok[j] ? silu_f(xv[j]) : 0.f;
            }
        }
        __syncthreads();
        *reinterpret_cast<float4*>(&Ys[lq][l4]) = make_float4(yv[0], yv[1], yv[2], yv[3]);
        *reinterpret_cast<float4*>(&Xs[lq][l4]) = make_float4(xv[0], xv[1], xv[2], xv[3]);
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            float4 a = *reinterpret_cast<const float4*>(&Ys[kk][ty * 4]);
            float4 b = *reinterpret_cast<const float4*>(&Xs[kk][tx * 4]);
            float aa[4] = {a.x, a.y, a.z, a.w}, bb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(aa[i], bb[j], acc[i][j]);
        }
    }
    const int taps = p.KH * p.KW;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int co = co0 + ty * 4 + i;
        if (co >= p.Cout || co >= p.CoutV) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int kf = kf0 + tx * 4 + j;
            if (kf >= p.Kf) continue;
            int tp = kf / p.Cin, c = kf - tp * p.Cin;
            if (c >= p.CinV) continue;
            atomicAdd(&p.dw[((int64_t)co * p.CinV + c) * taps + tp], acc[i][j]);
        }
    }
}

int wgrad_simt_launch(const ddpm_wgrad_args* a, cudaStream_t st) {
    WgP p;
    p.act = TV(a->act); p.dy = TV(a->dy); p.dw = a->dw;
    p.KH = a->KH; p.KW = a->KW; p.stride = a->stride; p.pad = a->pad; p.a_silu = a->a_silu;
    p.Cin = a->act.C; p.Cout = a->dy.C;
    p.CinV = a->cin_valid > 0 ? a->cin_valid : p.Cin; p.CoutV = a->cout_valid > 0 ? a->cout_valid : p.Cout;
    p.HoWo = a->dy.H * a->dy.W; p.Q = a->dy.N * p.HoWo; p.Kf = a->KH * a->KW * p.Cin;
    const int es = a->dtype == DDPM_F32 ? 4 : 2;
    p.vecA = (p.Cin % 4 == 0) && (a->act.pitch % 4 == 0) && al(a->act.ptr, 4 * es);
    p.vecY = (a->dy.pitch % 4 == 0) && al(a->dy.ptr, 4 * es);
    int tiles = ceil_div(p.Cout, BM) * ceil_div(p.Kf, BN);
    int splits = (148 * 4 + tiles - 1) / tiles;
    int maxs = ceil_div(p.Q, BK * 8);
    if (splits > maxs) splits = maxs;
    if (splits < 1) splits = 1;
    p.qper = ceil_div(ceil_div(p.Q, splits), BK) * BK;
    splits = ceil_div(p.Q, p.qper);
    dim3 grid(ceil_div(p.Cout, BM), ceil_div(p.Kf, BN), splits);
    if (a->dtype == DDPM_F32) CUDA_TRY(launch_kernel(wgrad_simt_kernel<float>, grid, dim3(CT), 0, st, p));
    else CUDA_TRY(launch_kernel(wgrad_simt_kernel<bf16>, grid, dim3(CT), 0, st, p));
    LAUNCH_OK();
    return 0;
}
