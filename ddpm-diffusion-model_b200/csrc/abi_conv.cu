// ddpm_conv / ddpm_conv_wgrad: argument validation and dispatch between the tcgen05 tensor-core
// kernels (conv_tc.cu, bf16 / fp16) and the CUDA-core kernels (conv_simt.cu, fp32 + every odd shape).
#include "common.cuh"

int conv_simt_launch(const ddpm_conv_args* a, cudaStream_t st);
int wgrad_simt_launch(const ddpm_wgrad_args* a, cudaStream_t st);
int conv_tc_supported(const ddpm_conv_args* a);
int conv_tc_launch(const ddpm_conv_args* a, cudaStream_t st);
int wgrad_tc_supported(const ddpm_wgrad_args* a);
int wgrad_tc_launch(const ddpm_wgrad_args* a, cudaStream_t st);

static int g_force_simt = 0;
extern "C" int ddpm_set_force_simt(int v) { g_force_simt = v; return 0; }
int ddpm_force_simt_flag() { return g_force_simt; }

extern "C" int ddpm_conv(const ddpm_conv_args* a, void* stream) {
    if (!a || !tensor_ok(&a->in) || !tensor_ok(&a->out) || !a->w) return DDPM_E_ARG;
    if (a->dtype != DDPM_F32 && a->dtype != DDPM_BF16 && a->dtype != DDPM_F16) return DDPM_E_ARG;
    if (a->KH <= 0 || a->KW <= 0 || a->stride <= 0 || a->pad < 0) return DDPM_E_ARG;
    if (a->in.N != a->out.N) return DDPM_E_ARG;
    if (a->mode == DDPM_CONV_NORMAL) {
        if (a->out.H != (a->in.H + 2 * a->pad - a->KH) / a->stride + 1) return DDPM_E_ARG;
        if (a->out.W != (a->in.W + 2 * a->pad - a->KW) / a->stride + 1) return DDPM_E_ARG;
    } else if (a->mode == DDPM_CONV_TRANSPOSED) {
        // out is the (larger) input-gradient; in is dY.  in.H must be the fwd conv's output size.
        if (a->in.H != (a->out.H + 2 * (a->KH - 1 - a->pad) - a->KH) / a->stride + 1) return DDPM_E_ARG;
    } else if (a->mode == DDPM_CONV_UP2X_PHASE) {
        // folded nearest-x2 + conv3x3: `in` is the low-resolution tensor, `out` the full-resolution view; tensor cores only
        if (a->out.H != 2 * a->in.H || a->out.W != 2 * a->in.W || a->KH != 2 || a->KW != 2 || a->stride != 1) return DDPM_E_ARG;
        if (a->up_phase < 0 || a->up_phase > 3 || a->res.ptr || a->z.ptr || a->in2.ptr || a->a_silu) return DDPM_E_ARG;
        if (!a->prefer_tc || g_force_simt || !conv_tc_supported(a)) return DDPM_E_ARG;
        return conv_tc_launch(a, (cudaStream_t)stream);
    } else return DDPM_E_ARG;
    if (a->res.ptr && (!tensor_ok(&a->res) || a->res.C != a->out.C || a->res.H != a->out.H || a->res.W != a->out.W)) return DDPM_E_ARG;
    if (a->z.ptr && (!tensor_ok(&a->z) || a->z.C != a->out.C || a->z.H != a->out.H || a->z.W != a->out.W)) return DDPM_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (a->in2.ptr) {
        if (!tensor_ok(&a->in2) || !a->w2 || a->mode != DDPM_CONV_NORMAL || a->stride != 1 || a->a_silu) return DDPM_E_ARG;
        if (a->in2.N != a->out.N || a->in2.H != a->out.H || a->in2.W != a->out.W) return DDPM_E_ARG;
        if (a->prefer_tc && !g_force_simt && conv_tc_supported(a)) return conv_tc_launch(a, st);      // one launch, K = 9*Cin + Cin2
        // every other path: the same sum as two launches (the 1x1 accumulates into the main result)
        ddpm_conv_args m = *a; m.in2.ptr = nullptr; m.w2 = nullptr;
        int rc = ddpm_conv(&m, stream); if (rc) return rc;
        ddpm_conv_args s2 = *a;
        s2.in = a->in2; s2.w = a->w2; s2.in2.ptr = nullptr; s2.w2 = nullptr;
        s2.KH = s2.KW = 1; s2.pad = 0; s2.bias = nullptr; s2.bias_n = 0; s2.tbias = nullptr; s2.res.ptr = nullptr; s2.z.ptr = nullptr;
        s2.epi = DDPM_EPI_ACCUM;
        return ddpm_conv(&s2, stream);
    }
    if (a->prefer_tc && !g_force_simt && conv_tc_supported(a)) return conv_tc_launch(a, st);
    return conv_simt_launch(a, st);
}

extern "C" int ddpm_conv_wgrad(const ddpm_wgrad_args* a, void* stream) {
    if (!a || !tensor_ok(&a->act) || !tensor_ok(&a->dy) || !a->dw) return DDPM_E_ARG;
    if (a->dtype != DDPM_F32 && a->dtype != DDPM_BF16 && a->dtype != DDPM_F16) return DDPM_E_ARG;
    if (a->KH <= 0 || a->KW <= 0 || a->stride <= 0 || a->pad < 0 || a->act.N != a->dy.N) return DDPM_E_ARG;
    if (a->dy.H != (a->act.H + 2 * a->pad - a->KH) / a->stride + 1) return DDPM_E_ARG;
    if (a->dy.W != (a->act.W + 2 * a->pad - a->KW) / a->stride + 1) return DDPM_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (a->prefer_tc && !g_force_simt && a->workspace && wgrad_tc_supported(a)) return wgrad_tc_launch(a, st);
    if (a->dbias) {                      // CUDA-core path: the bias gradient is a separate column sum of dy
        ddpm_tensor d = a->dy;
        if (a->cout_valid > 0) d.C = a->cout_valid;
        int rc = ddpm_colsum(&d, a->dtype, nullptr, a->dbias, stream);
        if (rc) return rc;
    }
    return wgrad_simt_launch(a, st);
}
