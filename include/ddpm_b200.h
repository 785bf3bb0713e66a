/*
 * ddpm_b200.h -- C ABI of libddpm_b200.so: the sm_100a CUDA implementation of the DDPM/DDIM hot
 * path of pablo-reyes8/ddpm-diffusion-model.
 *
 * The reference is pure Python/PyTorch and has no FFI of its own (SURVEY.md §8b); each entry point
 * below cites the reference site (path:line under /root/reference) whose ATen work it replaces.
 * INTEGRATION.md shows the ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns 0 on success, a positive cudaError_t, or a negative DDPM_E_* code;
 *   - no allocation, no host synchronisation, no hidden state except the schedule handle;
 *   - `stream` is a cudaStream_t passed as void*; all work is ordered on it (graph-capturable);
 *   - activations are NHWC with an optional zero halo of one pixel (struct ddpm_tensor), element
 *     type chosen by `dtype` (DDPM_F32 / DDPM_BF16 / DDPM_F16); parameters and their gradients are
 *     fp32 in the reference's OIHW / [out,in] layouts;
 *   - every entry point that accepts DDPM_BF16 accepts DDPM_F16 with the same shapes, the same
 *     paths (tcgen05 wherever bf16 takes the tensor cores) and the same semantics; any other dtype
 *     code returns DDPM_E_ARG.  fp32 -> fp16 conversions round to nearest and give +-inf beyond
 *     65504 (IEEE, as torch.autocast does), so a GradScaler sees the overflow in the fp32 gradients;
 *   - kernels never write the halo, so a buffer whose halo was zeroed once stays valid.
 */
#ifndef DDPM_B200_H
#define DDPM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DDPM_F32 0
#define DDPM_BF16 1
#define DDPM_F16 2   /* IEEE binary16 */

#define DDPM_E_ARG (-1)      /* invalid argument / unsupported shape */
#define DDPM_E_NOTREADY (-2) /* schedule handle not initialised */

/* NHWC view.  addr(n,y,x,c) = ptr + (((n*(H+2*halo) + y+halo)*(W+2*halo)) + x+halo)*pitch + c */
typedef struct {
    void* ptr;   /* element (n=0,y=-halo,x=-halo,c=0) of this view (channel offset folded in) */
    int32_t N, H, W, C;
    int32_t pitch; /* elements between consecutive pixels (>= C; > C for channel slices) */
    int32_t halo;  /* 0 or 1 */
} ddpm_tensor;

int ddpm_abi_version(void);
int ddpm_num_sms(int device, int* out);
/* Returns and resets the count of kernels this library launched since the last call. */
int64_t ddpm_launch_count(int reset);
/* Credits `n` kernel launches to the counter: a CUDA graph captured from these entry points launches the same kernels at
 * every replay without passing through the library (the host mirror adds the count it observed during capture). */
int ddpm_launch_count_add(int64_t n);
/* sizeof() of the six ABI structs in declaration order (ddpm_tensor, ddpm_conv_args, ddpm_lin_entry, ddpm_wgrad_args,
 * ddpm_pack_entry, ddpm_adam_hyper) so that a binding can verify its own layouts when it loads the library (the Python
 * mirror refuses to import on a mismatch).  Returns the number of entries written (<= n). */
int ddpm_abi_struct_sizes(int32_t* out, int n);

/* ---------------- schedule tables: difussion_class.py:46-68 (10 fp32 [T] buffers) ---------- */
/* rows: 0 betas 1 alphas 2 alphas_cumprod 3 sqrt_ac 4 sqrt_1m_ac 5 ac_prev 6 post_var
 *       7 post_logvar 8 post_coef1 9 post_coef2.   `tables_dev` is a device pointer [10][T]. */
int ddpm_schedule_create(const float* tables_dev, int T, int device, void** handle);
int ddpm_schedule_destroy(void* handle);

/* ---------------- diffusion elementwise: difussion_class.py:81-234 ------------------------ */
/* q_sample (:81-91).  x0, eps, xt: contiguous fp32 [B][chw]; t: int64 [B] (clamped to [0,T-1]). */
int ddpm_q_sample(void* sched, const float* x0, const float* eps, const int64_t* t, float* xt,
                  int B, int64_t chw, void* stream);
/* loss_simple tail (:113-116).  loss[0] += mean_b(w_b * mean_chw((noise-pred)^2)); caller zeroes
 * loss.  pred dtype f32/bf16/f16, contiguous [B][chw].  weight may be NULL. */
int ddpm_mse_fwd(const void* pred, int pred_dtype, const float* noise, const float* weight,
                 float* loss, int B, int64_t chw, void* stream);
/* d loss / d pred = 2 (pred-noise) w_b / (B*chw) * gout[0]; written in pred's dtype. */
int ddpm_mse_bwd(const void* pred, int pred_dtype, const float* noise, const float* weight,
                 const float* gout, void* dpred, int B, int64_t chw, void* stream);
/* per-sample max|x0_hat| before thresholding (:143).  amax: fp32 [B], zeroed by the call. */
int ddpm_x0_absmax(void* sched, const float* xt, const void* eps, int eps_dtype, const int64_t* t,
                   float* amax, int B, int64_t chw, void* stream);
/* flags for the sampler steps */
#define DDPM_CLAMP_X0 1   /* clamp x0_hat to [-1,1] (:150-151, :179-180) */
#define DDPM_DYN_THRESH 2 /* divide by max(amax,1).clamp(min=s) then clamp (:143-149) */
/* p_sample_step (:156-187) given eps_pred.  noise may be NULL only if all t == 0. */
int ddpm_p_sample_step(void* sched, const float* xt, const void* eps, int eps_dtype,
                       const float* noise, const int64_t* t, const float* amax, float dyn_s,
                       int flags, float* out, int B, int64_t chw, void* stream);
/* p_sample_step_ddim (:189-234) given eps_pred.  noise may be NULL when eta == 0. */
int ddpm_ddim_step(void* sched, const float* xt, const void* eps, int eps_dtype,
                   const float* noise, const int64_t* t, const int64_t* t_prev, float eta,
                   const float* amax, float dyn_s, int flags, float* out, int B, int64_t chw,
                   void* stream);
/* (clamp(x,-1,1)+1)/2: ddpm_inference.py:40, ddpim_inference.py:89 */
int ddpm_to_image01(const float* x, float* out, int64_t n, void* stream);
/* Sampler output path (SURVEY 8(f) f3): torchvision make_grid(nrow, padding, pad_value 0) of fp32 [N][C][H][W] images
 * in [0,1] (C = 1 or 3; one channel is replicated) and save_image's uint8 conversion trunc(clamp(v*255 + 0.5, 0, 255))
 * (ddpm_inference.py:41-45, ddpim_inference.py:90-93) in one pass.  grid_f32: [3][Hg][Wg] or NULL; grid_u8: [Hg][Wg][3]
 * (what PIL consumes) or NULL; Hg = (H+pad)*ceil(N/min(nrow,N)) + pad, Wg = (W+pad)*min(nrow,N) + pad; N == 1 returns the
 * image itself (Hg = H, Wg = W), like make_grid. */
int ddpm_image_grid(const float* x01, int N, int C, int H, int W, int nrow, int pad, float* grid_f32, uint8_t* grid_u8,
                    void* stream);

/* Input side (SURVEY 8(f) f4): one batch of a uint8 NHWC dataset resident in HBM -> fp32 NCHW in [-1,1], i.e.
 * transforms.ToTensor() + Normalize([0.5]*3,[0.5]*3) of src/data/load_data_local.py:90-95 / celebraHQ.py:40-43 for the
 * samples idx[0..B) (device int64; out of range is undefined behaviour -- the host side generates the permutation). */
int ddpm_batch_from_u8(const uint8_t* data, int64_t n_images, const int64_t* idx, int B, int H, int W, float* out,
                       void* stream);

/* ---------------- layout at the API boundary (NCHW-shaped, any strides <-> NHWC) ---------- */
/* dst->C may exceed src_C (channel padding for the tensor-core kernels): the extra channels are
 * written as zeros. */
int ddpm_nchw_to_nhwc(const void* src, int src_dtype, int src_C, int64_t sn, int64_t sc, int64_t sh,
                      int64_t sw, const ddpm_tensor* dst, int dst_dtype, void* stream);
int ddpm_nhwc_to_nchw(const ddpm_tensor* src, int src_dtype, void* dst, int dst_dtype, int64_t sn,
                      int64_t sc, int64_t sh, int64_t sw, void* stream);

/* ---------------- time embedding: attention.py:13-22 -------------------------------------- */
/* t: int64 or fp32 [B] (t_is_float); out: [B][dim] in `dtype`. */
int ddpm_sinusoid(const void* t, int t_is_float, int B, int dim, void* out, int dtype, void* stream);

/* ---------------- GroupNorm (+SiLU, +dropout): attention.py:38-39, unet_backbone.py:38,43 -- */
/* stats: double [N][G][2] = (sum, sum of squares) over the group's elements; zeroed by the call. */
int ddpm_gn_stats(const ddpm_tensor* x, int dtype, int groups, double* stats, void* stream);
/* out = drop(act(gn(x))); act: 0 none, 1 SiLU.  rng: device uint64[2] {seed, step} (may be NULL
 * when p_drop == 0); layer_id decorrelates call sites. */
int ddpm_gn_apply(const ddpm_tensor* x, int dtype, int groups, const double* stats, const float* gamma,
                  const float* beta, float eps, int act, float p_drop, const uint64_t* rng,
                  uint32_t layer_id, const ddpm_tensor* out, void* stream);
/* gn_stats + gn_apply in ONE launch: a thread-block cluster per image reduces the moments over
 * distributed shared memory, then re-reads the image (L2 hits) and writes `out`; `stats` is
 * written for the backward pass.  4 B/elem of HBM traffic (bf16) instead of 6. */
int ddpm_gn_fwd(const ddpm_tensor* x, int dtype, int groups, double* stats, const float* gamma,
                const float* beta, float eps, int act, float p_drop, const uint64_t* rng,
                uint32_t layer_id, const ddpm_tensor* out, void* stream);
/* backward of gn_apply, one launch (cluster per image; reduce, exchange, re-read from L2, write).
 * dx (+)= ...; dgamma/dbeta (fp32 [C]) are accumulated with atomics.  `ws` is unused (kept for
 * ABI stability; may be NULL).  dx may alias dy. */
int ddpm_gn_bwd(const ddpm_tensor* x, int dtype, int groups, const double* stats, const float* gamma,
                const float* beta, float eps, int act, float p_drop, const uint64_t* rng,
                uint32_t layer_id, const ddpm_tensor* dy, const ddpm_tensor* dx, int accumulate,
                float* dgamma, float* dbeta, float* ws, void* stream);

/* ddpm_gn_bwd that also emits the channel sums of the final dx: colsum_nc[n][c] (fp32, overwritten; may
 * be NULL) and colsum_c[c] += sum_n (may be NULL) -- the time-bias / conv-bias gradients of the layer that
 * produced x (unet_backbone.py:41,22), saving a separate ddpm_colsum pass over dx.
 * dy_scratch != 0: the caller no longer needs dy; the reduction phase leaves dz = dy*mask*act'(z) in it so
 * the second phase skips the mask / activation-derivative recomputation (dy's contents are then undefined). */
int ddpm_gn_bwd_colsum(const ddpm_tensor* x, int dtype, int groups, const double* stats, const float* gamma,
                       const float* beta, float eps, int act, float p_drop, const uint64_t* rng,
                       uint32_t layer_id, const ddpm_tensor* dy, const ddpm_tensor* dx, int accumulate,
                       float* dgamma, float* dbeta, float* colsum_nc, float* colsum_c, int dy_scratch, void* stream);

/* nearest x2 (unet_backbone.py:63) and its adjoint (2x2 sum) */
int ddpm_upsample2x(const ddpm_tensor* x, const ddpm_tensor* out, int dtype, void* stream);
int ddpm_upsample2x_bwd(const ddpm_tensor* dy, const ddpm_tensor* dx, int dtype, int accumulate, void* stream);
/* out[n,2y,2x] = x[n,y,x], zeros elsewhere (whole interior written): turns the data / weight gradient
 * of a stride-2 convolution into stride-1 problems for the tensor-core kernels */
int ddpm_zero_upsample2x(const ddpm_tensor* x, const ddpm_tensor* out, int dtype, void* stream);
/* out = a + b (all three may alias channel slices); used for gradient fan-in */
int ddpm_add(const ddpm_tensor* a, const ddpm_tensor* b, const ddpm_tensor* out, int dtype, void* stream);
/* out_nc[n][c] = sum_pixels dy (fp32, overwritten, may be NULL); dbias[c] += sum_n (may be NULL) */
int ddpm_colsum(const ddpm_tensor* dy, int dtype, float* out_nc, float* dbias, void* stream);

/* ---------------- convolution / linear as implicit GEMM ----------------------------------- */
/* nn.Conv2d 3x3 s1/s2 p1, 1x1 (unet_backbone.py:22,32,35,51,60,97,100; attention.py:53-54) and
 * nn.Linear as a 1x1 conv on H=W=1 (attention.py:30,32; unet_backbone.py:27). */
#define DDPM_CONV_NORMAL 0
#define DDPM_CONV_TRANSPOSED 1 /* gather for the data-gradient of a strided conv */
#define DDPM_CONV_UP2X_PHASE 2 /* one output phase of `conv3x3(nearest_upsample_x2(in))` (unet_backbone.py:63-64) computed straight
                                * from the LOW-resolution input: out[n, 2y+py, 2x+px] = bias + sum over a 2x2 neighbourhood of
                                * in[n, y+ty+py-1, x+tx+px-1] with the phase's pre-summed weights (ddpm_pack_weights_up2x).
                                * `in` is [N,H,W,Cin], `out` the [N,2H,2W,Cout] view; KH = KW = 2, stride 1, up_phase = 2*py+px.
                                * Four calls cover the output: 16 instead of 36 multiply-adds per low-resolution pixel pair
                                * and the up-sampled tensor is never materialised.  Tensor-core path (bf16 / fp16) only. */
#define DDPM_EPI_ACCUM 1       /* out += result (in place; gradient fan-in, residual) */
#define DDPM_EPI_DSILU 2       /* result *= silu'(z[n,c])  (time path backward) */
typedef struct {
    ddpm_tensor in;        /* activations (or dY for dgrad) */
    ddpm_tensor out;       /* result view (may be a channel slice of a wider buffer) */
    const void* w;         /* packed weights [Cout][KH*KW][Cin] in `dtype` (see ddpm_pack_weights) */
    const float* bias;     /* fp32 [bias_n] or NULL */
    const float* tbias;    /* per-image bias fp32 [N][tbias_pitch] or NULL (time_proj output; the time path is fp32) */
    int32_t tbias_pitch;
    ddpm_tensor res;       /* residual added in the epilogue; res.ptr == NULL for none */
    ddpm_tensor z;         /* pre-activation for DDPM_EPI_DSILU; z.ptr == NULL for none */
    int32_t KH, KW, stride, pad;
    int32_t mode;          /* DDPM_CONV_NORMAL / DDPM_CONV_TRANSPOSED */
    int32_t a_silu;        /* apply SiLU to the input operand on load (time path) */
    int32_t epi;           /* DDPM_EPI_* flags */
    int32_t dtype;
    int32_t prefer_tc;     /* 1: use the tcgen05 kernel when the shape qualifies (bf16 / fp16 only) */
    int32_t bias_n;        /* entries in `bias` (0: out.C); fewer when out carries zero-padded channels */
    /* Optional second operand: out = conv(in; w) + conv1x1(in2; w2) (+ bias ...), i.e. the ResBlock's `conv2(h) + skip(x)`
     * (unet_backbone.py:35,46) as ONE implicit GEMM whose K dimension is 9*Cin + Cin2.  in2 has the geometry of `out`
     * (stride-1 main conv); w2 is packed [Cout][1][Cin2].  in2.ptr == NULL: none. */
    ddpm_tensor in2;
    const void* w2;
    int32_t up_phase;      /* DDPM_CONV_UP2X_PHASE: 2*py + px in 0..3 (ignored otherwise) */
} ddpm_conv_args;
int ddpm_conv(const ddpm_conv_args* a, void* stream);
/* test / tuning hooks: force the CUDA-core kernels */
int ddpm_set_force_simt(int on);
/* Force tensor-core paths that the planners otherwise pick only for other shapes (tests, A/B measurements).  Bit 0 of
 * `mode` must be 1, bits 1-3 and base_offset must be 0, and mode >> 4 is a combination of
 *   32    convolution: keep a channel tile wider than 128 (NT = 192 / 256) instead of halving it
 *   64    convolution: stream the weights with every stage instead of keeping them resident in shared memory
 *   128   convolution: 16-byte instead of 32-byte epilogue loads / stores
 *   1024  weight gradient: the single-CTA kernel instead of the CTA-pair kernel
 * (1 restores the default planning).  The flags are read on the host when a call plans its launch; no kernel sees them.
 * Anything else returns DDPM_E_ARG and leaves the setting unchanged. */
int ddpm_set_tc_mode(int mode, int base_offset);

/* All time_proj linears of a UNet in one launch (unet_backbone.py:25-27,41): out[m][col0_i + n] =
 * sum_k f(x[m][k]) W_i[n][k] + b_i[n], f = SiLU when a_silu.  `entries_dev` is an array in DEVICE memory. */
typedef struct {
    const float* w;      /* fp32 [N][K] (the nn.Linear weight itself) */
    const float* bias;   /* fp32 [N] or NULL */
    int32_t N, col0;     /* output features; first output column in `out` */
    const float* bias2;  /* optional second fp32 [N] bias added as well: the bias of the convolution that consumes this
                          * time bias (unet_backbone.py:40-41), so that its epilogue adds ONE per-image vector */
} ddpm_lin_entry;
int ddpm_linear_grouped_fwd(const float* x, int M, int K, int xpitch, const ddpm_lin_entry* entries_dev, int n,
                            int max_N, float* out, int out_pitch, int a_silu, void* stream);
/* Backward of one time_proj in one launch: dw[N][K] += dy^T silu(temb), db[N] += colsum(dy) (db may be NULL),
 * dtemb[B][K] (+)= (dy W) * silu'(temb).  dy is [B][N] with row pitch dy_pitch. */
int ddpm_time_proj_bwd(const float* temb, int B, int K, const float* dy, int dy_pitch, int N, const float* w,
                       float* dw, float* db, float* dtemb, int accum_dtemb, void* stream);

typedef struct {
    ddpm_tensor act;   /* forward input operand of the conv */
    ddpm_tensor dy;    /* gradient of the conv output */
    float* dw;         /* fp32 OIHW [Cout][Cin][KH][KW], accumulated */
    int32_t KH, KW, stride, pad;
    int32_t a_silu;
    int32_t dtype;
    int32_t prefer_tc;
    void* workspace;          /* split-K partials for the tensor-core kernel (may be NULL -> CUDA cores) */
    int64_t workspace_bytes;
    int32_t cin_valid, cout_valid; /* >0: act / dy carry zero-padded channels; dw is [cout_valid][cin_valid][KH][KW] */
    float* dbias;             /* fp32 [cout_valid or dy.C], accumulated with sum over pixels of dy (conv bias gradient); may be NULL.
                               * The tensor-core kernel gets it from one extra N=16 MMA per K-step against a tile of ones. */
} ddpm_wgrad_args;
int ddpm_conv_wgrad(const ddpm_wgrad_args* a, void* stream);
/* bytes of workspace the tensor-core wgrad wants for this problem (0: it will not be used) */
int64_t ddpm_wgrad_workspace_bytes(const ddpm_wgrad_args* a);

/* fp32 OIHW -> [Cout_pad][KH*KW][Cin_pad] (fwd) and flipped/transposed [Cin_pad][KH*KW][Cout_pad]
 * (dgrad); padded rows/columns are zero.  cin_pad / cout_pad <= 0 mean "no padding". */
int ddpm_pack_weights(const float* w, int Cout, int Cin, int KH, int KW, void* w_fwd, void* w_dgrad,
                      int dtype, int cin_pad, int cout_pad, void* stream);

/* Phase weights of the folded `nearest x2 up-sample + conv3x3` (DDPM_CONV_UP2X_PHASE): out[ph][co][t][ci] (ph = 2*py+px,
 * t = 2*ty+tx) = sum of w[co][ci][ky][kx] over ky in S(py,ty), kx in S(px,tx) with S(0,0)={0}, S(0,1)={1,2}, S(1,0)={0,1},
 * S(1,1)={2} -- summed in fp32, then rounded to `dtype`.  w is fp32 OIHW [Cout][Cin][3][3] (unet_backbone.py:60). */
int ddpm_pack_weights_up2x(const float* w, int Cout, int Cin, void* out, int dtype, void* stream);

/* the same for many weights in one launch; `entries_dev` is an array in DEVICE memory */
typedef struct {
    const float* w;      /* fp32 OIHW source */
    void* wf;            /* packed fprop copy or NULL */
    void* wd;            /* packed dgrad copy or NULL */
    int32_t Cout, Cin, taps, CiP, CoP, dtype;
} ddpm_pack_entry;
/* An entry whose dtype is not DDPM_F32 / DDPM_BF16 / DDPM_F16 is skipped (the entries are in device memory). */
int ddpm_pack_weights_batched(const ddpm_pack_entry* entries_dev, int n, void* stream);

/* ---------------- attention: attention.py:56-74 -------------------------------------------- */
/* qkv: NHWC with channel = s*heads*d + head*d + i (s in q,k,v) -- the layout conv `qkv` emits, so
 * the four permute+contiguous copies (:63-65,72) disappear.  lse: fp32 [N][heads][H*W]. */
int ddpm_attn_fwd(const ddpm_tensor* qkv, const ddpm_tensor* out, int heads, int d, float* lse,
                  int dtype, void* stream);
/* scratch: ddpm_attn_bwd_scratch_floats(qkv, out, ...) fp32 elements.  When qkv / out take the tensor-core kernels, dout
 * and dqkv must too (same geometry, 16-byte aligned, pitch a multiple of 8) and dout->halo must equal qkv->halo;
 * otherwise the call returns DDPM_E_ARG and writes nothing. */
int ddpm_attn_bwd(const ddpm_tensor* qkv, const ddpm_tensor* out, const ddpm_tensor* dout,
                  const float* lse, const ddpm_tensor* dqkv, int heads, int d, float* scratch,
                  int dtype, void* stream);
/* fp32 elements of `scratch` ddpm_attn_bwd needs for this problem, from qkv / out alone: N*N-sized P and dS matrices
 * ([N][heads][HW][HW] * 2) for the CUDA-core kernels, one value per (image, head, query) for the tensor-core kernels
 * (bf16 / fp16, head_dim 32 / 64 / 128, W <= 128, any H; 16-byte aligned, pitch a multiple of 8), which recompute P from the
 * forward's log-sum-exp. */
int64_t ddpm_attn_bwd_scratch_floats(const ddpm_tensor* qkv, const ddpm_tensor* out, int heads, int d, int dtype);

/* ---------------- optimiser-side parameter pass -------------------------------------------- */
/* train_one_epoch.py:94-115 + ema.py:15-23 over flat fp32 arenas.
 * stats: fp32 [4] = {sum g^2 (of the still-scaled grads), found_inf flag, -, -}; zeroed by reduce. */
int ddpm_param_reduce(const float* grad, int64_t n, float* stats, void* stream);
typedef struct {
    float lr, beta1, beta2, eps, weight_decay;
    float max_norm;     /* <= 0: no clipping */
    float ema_decay;    /* used when ema != NULL */
    int32_t adamw;      /* 1: decoupled decay (AdamW); 0: L2 into the gradient (Adam) */
} ddpm_adam_hyper;
/* step: device fp32 [1], incremented when no inf was found (AdamW `state["step"]`).
 * scale: the GradScaler's device `_scale` fp32 [1], or NULL for 1.0.
 * One pass: g*=1/scale, clip by global norm, Adam(W) update, EMA lerp.  When found_inf, p/m/v are
 * left untouched (GradScaler.step skip) but the EMA still moves (ema.update is unconditional). */
int ddpm_param_update(float* p, const float* g, float* m, float* v, float* ema, int64_t n,
                      const float* stats, float* step, const float* scale, const ddpm_adam_hyper* h,
                      void* stream);
/* GradScaler.update() on its own tensors: scale *= backoff on inf, *= growth after `interval`
 * clean steps (tracker: int32 [1]).  Also records stats[2] = the scale before the update (the one this
 * step's gradients carried), so a later grad-norm read-back divides by the right factor. */
int ddpm_scaler_update(float* scale, int32_t* tracker, float* stats, float growth, float backoff,
                       int interval, void* stream);
/* For optimisers other than Adam(W): g *= clip/scale in place (g = 0 when inf was found). */
int ddpm_grad_unscale_clip(float* g, int64_t n, const float* stats, const float* scale, float max_norm,
                           void* stream);
/* EMA only (any optimiser): shadow = d*shadow + (1-d)*p */
int ddpm_ema_update(float* shadow, const float* p, int64_t n, float decay, void* stream);
/* rng[1] += 1 (dropout stream position), graph-capturable */
int ddpm_rng_advance(uint64_t* rng, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DDPM_B200_H */
