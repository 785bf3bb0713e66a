"""Drop-in for src/model/difussion_class.py: same constructor, buffers and methods; q_sample, the
MSE loss, the DDPM step and the DDIM step each run as ONE fused CUDA kernel reading the schedule
from __constant__ memory (the reference issues 46 / 76 / 118 ATen calls, SURVEY.md §2.2 row 11)."""
import ctypes as C
from typing import Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import _lib
from .difussion_utils import ScheduleKind, beta_schedule_cosine, beta_schedule_linear, extract

TABLE_ORDER = ("betas", "alphas", "alphas_cumprod", "sqrt_alphas_cumprod", "sqrt_one_minus_alphas_cumprod",
               "alphas_cumprod_prev", "posterior_variance", "posterior_log_variance",
               "posterior_mean_coef1", "posterior_mean_coef2")


def _dt(x: torch.Tensor) -> int:
    if x.dtype == torch.float32:
        return _lib.F32
    if x.dtype == torch.bfloat16:
        return _lib.BF16
    if x.dtype == torch.float16:
        return _lib.F16
    raise TypeError(f"ddpm_b200: unsupported tensor dtype {x.dtype} (fp32 / bf16 / fp16 only)")


def _f32c(x: torch.Tensor) -> torch.Tensor:
    if x.dtype != torch.float32:
        x = x.float()
    return x if x.is_contiguous() else x.contiguous()


def _cuda_only(x: torch.Tensor, what: str):
    if not x.is_cuda:
        raise RuntimeError(f"ddpm_b200.Diffusion.{what}: tensors are on '{x.device}'; this implementation "
                           "is CUDA-only (sm_100a) and has no CPU fallback")


def _stream(x: torch.Tensor) -> int:
    return _lib.stream_for(x.device)


class _MSE(torch.autograd.Function):
    """loss = mean_b(w_b * mean_chw((noise - pred)^2))  (difussion_class.py:113-116)."""

    @staticmethod
    def forward(ctx, pred, noise, weight):
        pred_c = pred if pred.is_contiguous() else pred.contiguous()
        B = pred_c.shape[0]
        chw = pred_c.numel() // B
        loss = torch.zeros((), dtype=torch.float32, device=pred.device)
        _lib.call("ddpm_mse_fwd", pred_c.data_ptr(), _dt(pred_c), noise.data_ptr(),
                  weight.data_ptr() if weight is not None else None, loss.data_ptr(), B, chw, _stream(pred))
        ctx.save_for_backward(pred_c, noise, weight)
        return loss

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gout):
        pred, noise, weight = ctx.saved_tensors
        B = pred.shape[0]
        chw = pred.numel() // B
        g = _f32c(gout)
        dpred = torch.empty_like(pred)
        _lib.call("ddpm_mse_bwd", pred.data_ptr(), _dt(pred), noise.data_ptr(),
                  weight.data_ptr() if weight is not None else None, g.data_ptr(), dpred.data_ptr(), B, chw,
                  _stream(pred))
        return dpred, None, None


class Diffusion(nn.Module):
    """difussion_class.py:10-234."""

    def __init__(self, T: int = 1000, schedule: ScheduleKind = "linear", beta_min: float = 1e-4,
                 beta_max: float = 2e-2, cosine_s: float = 0.008, clamp_x0: bool = True,
                 dynamic_threshold: Optional[float] = None, img_size=None):
        super().__init__()
        self.T = int(T)
        self.clamp_x0 = clamp_x0
        self.dynamic_threshold = dynamic_threshold
        self.img_size = img_size
        if schedule == "linear":
            betas = beta_schedule_linear(T, beta_min, beta_max)
        elif schedule == "cosine":
            betas = beta_schedule_cosine(T, s=cosine_s)
        else:
            raise ValueError(f"schedule desconocido: {schedule}")
        # difussion_class.py:43-68 -- identical op order => identical bits
        alphas = 1.0 - betas
        ac = torch.cumprod(alphas, dim=0)
        ac_prev = F.pad(ac[:-1], (1, 0), value=1.0)
        post_var = betas * (1.0 - ac_prev) / (1.0 - ac)
        tables = {
            "betas": betas, "alphas": alphas, "alphas_cumprod": ac,
            "sqrt_alphas_cumprod": torch.sqrt(ac),
            "sqrt_one_minus_alphas_cumprod": torch.sqrt(1.0 - ac),
            "alphas_cumprod_prev": ac_prev,
            "posterior_variance": post_var.clamp(min=1e-20),
            "posterior_log_variance": torch.log(post_var.clamp(min=1e-20)),
            "posterior_mean_coef1": betas * torch.sqrt(ac_prev) / (1.0 - ac),
            "posterior_mean_coef2": (1.0 - ac_prev) * torch.sqrt(alphas) / (1.0 - ac),
        }
        for name in TABLE_ORDER:
            self.register_buffer(name, tables[name], persistent=False)   # state_dict stays empty
        self._sched = {}     # device -> (stacked [10][T] tensor, C handle, fingerprint)

    # ------------------------------------------------------------------ schedule handle
    def _handle(self, device) -> int:
        key = str(device)
        fp = tuple(int(getattr(self, n)._version) for n in TABLE_ORDER)
        ent = self._sched.get(key)
        if ent is not None and ent[2] == fp:
            return ent[1]
        if ent is not None:
            _lib.call("ddpm_schedule_destroy", ent[1])
        stacked = torch.stack([getattr(self, n).detach().to(device=device, dtype=torch.float32) for n in TABLE_ORDER]).contiguous()
        h = C.c_void_p()
        _lib.call("ddpm_schedule_create", stacked.data_ptr(), self.T, torch.device(device).index or 0, C.byref(h))
        self._sched[key] = (stacked, h.value, fp)
        return h.value

    def __del__(self):
        try:
            for _, h, _ in self._sched.values():
                _lib.lib.ddpm_schedule_destroy(h)
        except Exception:
            pass

    @staticmethod
    def _t64(t: torch.Tensor, device) -> torch.Tensor:
        """int64 timesteps on `device` (float t is truncated like extract's .long())."""
        if t.dtype != torch.int64 or t.device != device:
            t = t.to(device=device, dtype=torch.int64)
        return t if t.is_contiguous() else t.contiguous()

    # ------------------------------------------------------------------ q(x_t | x_0)
    def sample_timesteps(self, batch_size: int, device=None) -> torch.Tensor:
        """difussion_class.py:72-78: t ~ U{1..T-1} (t = 0 is never trained)."""
        if device is None:
            device = self.betas.device
        return torch.randint(1, self.T, (batch_size,), device=device, dtype=torch.long)

    @torch.no_grad()
    def q_sample(self, x0: torch.Tensor, t: torch.Tensor, eps: Optional[torch.Tensor] = None) -> torch.Tensor:
        """difussion_class.py:81-91: x_t = sqrt(ab_t) x0 + sqrt(1-ab_t) eps, one kernel.
        (Not differentiable w.r.t. x0/eps -- nothing on the reference's path needs that.)"""
        _cuda_only(x0, "q_sample")
        if eps is None:
            eps = torch.randn_like(x0)
        x0c, ec = _f32c(x0), _f32c(eps)
        out = torch.empty_like(x0c)
        B = x0c.shape[0]
        _lib.call("ddpm_q_sample", self._handle(x0.device), x0c.data_ptr(), ec.data_ptr(),
                  self._t64(t, x0.device).data_ptr(), out.data_ptr(), B, x0c.numel() // B, _stream(x0))
        return out

    def loss_simple(self, model_eps_pred_fn, x0: torch.Tensor, t: torch.Tensor,
                    noise: Optional[torch.Tensor] = None, weight: Optional[torch.Tensor] = None) -> torch.Tensor:
        """difussion_class.py:95-116.  RNG order preserved: randn_like(x0) is drawn here."""
        _cuda_only(x0, "loss_simple")
        if noise is None:
            noise = torch.randn_like(x0)
        noise_c = _f32c(noise)
        x_t = self.q_sample(x0, t, eps=noise_c)
        if x0.dim() == 4 and x0.is_contiguous(memory_format=torch.channels_last) and not x0.is_contiguous():
            x_t = x_t.contiguous(memory_format=torch.channels_last)
        eps_pred = model_eps_pred_fn(x_t, t)
        if eps_pred.dtype not in (torch.float32, torch.bfloat16, torch.float16):
            eps_pred = eps_pred.float()
        w = _f32c(weight) if weight is not None else None
        return _MSE.apply(eps_pred, noise_c, w)

    # ------------------------------------------------------------------ posterior helpers
    def posterior_mean_variance(self, x_t: torch.Tensor, x0_hat: torch.Tensor, t: torch.Tensor):
        """difussion_class.py:120-130 (public helper; the sampler kernels fuse this)."""
        c1 = extract(self.posterior_mean_coef1, t, x_t.shape)
        c2 = extract(self.posterior_mean_coef2, t, x_t.shape)
        return (c1 * x0_hat + c2 * x_t, extract(self.posterior_variance, t, x_t.shape),
                extract(self.posterior_log_variance, t, x_t.shape))

    def _flags_amax(self, x_t, eps, t64, extra_clip: bool):
        flags, amax, s = 0, None, 0.0
        if self.dynamic_threshold is not None:
            flags |= _lib.DYN_THRESH
            s = float(self.dynamic_threshold)
            B = x_t.shape[0]
            amax = torch.empty(B, dtype=torch.float32, device=x_t.device)
            _lib.call("ddpm_x0_absmax", self._handle(x_t.device), x_t.data_ptr(), eps.data_ptr(), _dt(eps),
                      t64.data_ptr(), amax.data_ptr(), B, x_t.numel() // B, _stream(x_t))
        elif self.clamp_x0 or extra_clip:
            flags |= _lib.CLAMP_X0
        return flags, amax, s

    @torch.no_grad()
    def predict_x0(self, x_t: torch.Tensor, eps_pred: torch.Tensor, t: torch.Tensor) -> torch.Tensor:
        """difussion_class.py:132-152, as a DDIM step onto t_prev with ab_prev = 1 is not available for
        every schedule, this helper evaluates the formula with the per-sample coefficients directly."""
        _cuda_only(x_t, "predict_x0")
        sa = extract(self.sqrt_alphas_cumprod, t.clone(), x_t.shape)
        so = extract(self.sqrt_one_minus_alphas_cumprod, t.clone(), x_t.shape)
        x0 = (x_t - so * eps_pred) / (sa + 1e-12)
        if self.dynamic_threshold is not None:
            amax = x0.abs().flatten(1).max(dim=1).values.clamp(min=1.0).clamp(min=self.dynamic_threshold)
            x0 = (x0 / amax.view(-1, *([1] * (x0.dim() - 1)))).clamp(-1, 1)
        elif self.clamp_x0:
            x0 = x0.clamp(-1, 1)
        return x0

    # ------------------------------------------------------------------ samplers' single steps
    @torch.no_grad()
    def p_sample_step(self, model_eps_pred_fn, x_t: torch.Tensor, t: torch.Tensor, eta: float = 1.0,
                      use_ema_model: bool = True, clip_x0: Optional[bool] = None,
                      noise: Optional[torch.Tensor] = None) -> torch.Tensor:
        """difussion_class.py:156-187.  `eta` and `use_ema_model` are ignored, as in the reference."""
        _cuda_only(x_t, "p_sample_step")
        if clip_x0 is None:
            clip_x0 = self.clamp_x0
        eps = model_eps_pred_fn(x_t, t)
        if eps.dtype not in (torch.float32, torch.bfloat16, torch.float16):
            eps = eps.float()
        eps = eps if eps.is_contiguous() else eps.contiguous()
        x = _f32c(x_t)
        t64 = self._t64(t, x.device)
        flags, amax, s = self._flags_amax(x, eps, t64, bool(clip_x0))
        if noise is None:
            noise = torch.randn_like(x_t)
        z = _f32c(noise)
        out = torch.empty_like(x)
        B = x.shape[0]
        _lib.call("ddpm_p_sample_step", self._handle(x.device), x.data_ptr(), eps.data_ptr(), _dt(eps),
                  z.data_ptr(), t64.data_ptr(), amax.data_ptr() if amax is not None else None, s, flags,
                  out.data_ptr(), B, x.numel() // B, _stream(x))
        return out

    @torch.no_grad()
    def p_sample_step_ddim(self, model_eps_pred_fn, x_t: torch.Tensor, t: torch.Tensor, t_prev: torch.Tensor,
                           eta: float = 0.0, clip_x0: Optional[bool] = None,
                           noise: Optional[torch.Tensor] = None) -> torch.Tensor:
        """difussion_class.py:189-234.  Noise is drawn even when eta == 0 (RNG-stream parity, App. C.5)
        but the kernel skips reading it then (sigma*z is exactly 0)."""
        _cuda_only(x_t, "p_sample_step_ddim")
        if clip_x0 is None:
            clip_x0 = self.clamp_x0
        if noise is None:
            noise = torch.randn_like(x_t)
        eps = model_eps_pred_fn(x_t, t)
        if eps.dtype not in (torch.float32, torch.bfloat16, torch.float16):
            eps = eps.float()
        eps = eps if eps.is_contiguous() else eps.contiguous()
        x = _f32c(x_t)
        t64, tp64 = self._t64(t, x.device), self._t64(t_prev, x.device)
        flags, amax, s = self._flags_amax(x, eps, t64, bool(clip_x0))
        z = _f32c(noise)
        out = torch.empty_like(x)
        B = x.shape[0]
        _lib.call("ddpm_ddim_step", self._handle(x.device), x.data_ptr(), eps.data_ptr(), _dt(eps),
                  z.data_ptr(), t64.data_ptr(), tp64.data_ptr(), float(eta),
                  amax.data_ptr() if amax is not None else None, s, flags, out.data_ptr(), B,
                  x.numel() // B, _stream(x))
        return out


def to_image01(x: torch.Tensor) -> torch.Tensor:
    """(clamp(x,-1,1)+1)/2 -- ddpm_inference.py:40 / ddpim_inference.py:89 as one kernel."""
    _cuda_only(x, "to_image01")
    xc = _f32c(x)
    out = torch.empty_like(xc)
    _lib.call("ddpm_to_image01", xc.data_ptr(), out.data_ptr(), xc.numel(), _stream(xc))
    return out
