"""torch.autograd bridges between the reference-shaped nn.Modules and the engine.

One autograd node per *module call* (whole UNet, or a ResBlock / AttnBlock / Downsample / Upsample
/ TimeMLP used on its own).  Parameter gradients are accumulated by the kernels straight into
`param.grad` (fp32, created zeroed on first use), so backward returns None for them; the parameters
are still passed to `apply` so autograd knows the output depends on them.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib, engine

_RNG = {}        # device -> int64[2] tensor {seed, step} for the dropout Philox stream


def rng_state(device) -> torch.Tensor:
    key = str(device)
    st = _RNG.get(key)
    if st is None:
        st = torch.tensor([torch.initial_seed() & 0x7FFFFFFFFFFFFFFF, 0], dtype=torch.int64, device=device)
        _RNG[key] = st
    return st


def seed_dropout(seed: int, device) -> None:
    """Re-seed the dropout stream (statistical, not bitwise, parity with ATen's Philox; SURVEY §7)."""
    _RNG[str(device)] = torch.tensor([seed & 0x7FFFFFFFFFFFFFFF, 0], dtype=torch.int64, device=device)


def _require_cuda(x: torch.Tensor, what: str) -> None:
    if not x.is_cuda:
        raise RuntimeError(
            f"ddpm_b200.{what}: input is on '{x.device}'. This implementation is CUDA-only (sm_100a) and has "
            "no CPU fallback; move the module and its inputs to a B200.")


def compute_dtype(x: torch.Tensor) -> tuple:
    """(engine dtype code, dtype of the returned tensor) following the reference's autocast policy:
    bf16 / fp16 autocast -> activations and result in that dtype (conv/linear are autocast-to-lower-precision
    ops, unet_backbone.py:215 ends in a conv); outside autocast a bf16 / fp16 input runs in its own dtype;
    otherwise fp32."""
    if torch.is_autocast_enabled("cuda"):
        adt = torch.get_autocast_dtype("cuda")
        if adt == torch.bfloat16:
            return _lib.BF16, torch.bfloat16
        if adt == torch.float16:
            return _lib.F16, torch.float16
        raise NotImplementedError(f"ddpm_b200 supports bf16 and fp16 autocast, not {adt}")
    if x.dtype == torch.bfloat16:
        return _lib.BF16, torch.bfloat16
    if x.dtype == torch.float16:
        return _lib.F16, torch.float16
    return _lib.F32, torch.float32


def make_exec(x: torch.Tensor, module: torch.nn.Module, need_grad: bool) -> engine.Exec:
    dt, _ = compute_dtype(x)
    shared = rng_state(x.device)
    E = engine.Exec(x.device, dt, module.training, need_grad, rng=shared)
    if module.training:
        _lib.call("ddpm_rng_advance", shared.data_ptr(), E.stream)
        # The dropout masks of THIS call are a function of {seed, step} as they are now.  Backward rebuilds the masks from
        # E.rng, so it must see this call's step, not whatever the shared counter has advanced to by then (a second
        # training-mode forward before backward: chained stand-alone ResBlocks, two model(x) calls summed, a no_grad
        # forward in between).  A 16-byte device-side snapshot per call, stream-ordered after the advance.
        E.rng = shared.clone()
    return E


def _needs_grad(module: torch.nn.Module, *inputs) -> bool:
    if not torch.is_grad_enabled():
        return False
    if any(isinstance(i, torch.Tensor) and i.requires_grad for i in inputs):
        return True
    return any(p.requires_grad for p in module.parameters())


class _UNetFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, E, out_dtype, x, t, *params):
        out, saved = engine.unet_forward(E, model, x, t, out_dtype)
        ctx.model, ctx.E, ctx.saved = model, E, saved
        ctx.need_dx = x.requires_grad
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dy):
        saved, ctx.saved = ctx.saved, None
        if saved is None:
            raise RuntimeError("ddpm_b200: backward through a UNet call made without grad")
        dx = engine.unet_backward(ctx.E, ctx.model, saved, dy, ctx.need_dx)
        return (None, None, None, dx, None) + (None,) * (len(ctx.needs_input_grad) - 5)


def unet_apply(model, x: torch.Tensor, t: torch.Tensor) -> torch.Tensor:
    _require_cuda(x, "UNetDenoiser")
    need = _needs_grad(model, x)
    E = make_exec(x, model, need)
    _, out_dtype = compute_dtype(x)
    if not need:
        out, _ = engine.unet_forward(E, model, x, t, out_dtype)
        return out
    return _UNetFn.apply(model, E, out_dtype, x, t, *[p for p in model.parameters() if p.requires_grad])


class _BlockFn(torch.autograd.Function):
    """Generic single-module node.  `fwd(E, *acts_or_tensors) -> (out tensor, saved)` and
    `bwd(E, saved, dy) -> tuple of input grads` are supplied by the caller."""

    @staticmethod
    def forward(ctx, fwd, bwd, E, n_in, *args):
        ins = args[:n_in]
        out, saved = fwd(E, *ins)
        ctx.bwd, ctx.E, ctx.saved, ctx.n_in, ctx.n_args = bwd, E, saved, n_in, len(args)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dy):
        saved, ctx.saved = ctx.saved, None
        grads = ctx.bwd(ctx.E, saved, dy)
        grads = tuple(grads) + (None,) * (ctx.n_in - len(grads))
        return (None, None, None, None) + grads + (None,) * (ctx.n_args - ctx.n_in)


def block_apply(module, fwd, bwd, *inputs):
    need = _needs_grad(module, *inputs)
    E = make_exec(inputs[0], module, need)
    if not need:
        return fwd(E, *inputs)[0]
    return _BlockFn.apply(fwd, bwd, E, len(inputs), *inputs, *[p for p in module.parameters() if p.requires_grad])


# ---------------------------------------------------------------------------------------------
# stand-alone module calls
# ---------------------------------------------------------------------------------------------
def resblock_apply(blk, x: torch.Tensor, t_emb: torch.Tensor) -> torch.Tensor:
    _require_cuda(x, "ResBlock")
    _, out_dtype = compute_dtype(x)

    def fwd(E, x_, temb_):
        temb32 = temb_.float().contiguous()
        tb = engine.linear_fwd(E, temb32, blk.time_proj[1], True)
        xa = engine.to_nhwc(E, x_)
        out, sv = engine.resblock_fwd(E, blk, xa, tb, None, 1)
        return engine.to_nchw(E, out, out_dtype), (sv, temb32)

    def bwd(E, saved, dy):
        sv, temb32 = saved
        dx, dtb = engine.resblock_bwd(E, blk, sv, engine.to_nhwc(E, dy))
        dtemb = engine.linear_bwd(E, temb32, blk.time_proj[1], True, dtb, None, False)
        return engine.to_nchw(E, dx, x.dtype if x.dtype in (torch.float32, torch.bfloat16, torch.float16) else torch.float32), dtemb.to(t_emb.dtype)

    return block_apply(blk, fwd, bwd, x, t_emb)


def attn_apply(blk, x: torch.Tensor) -> torch.Tensor:
    _require_cuda(x, "AttnBlock")
    _, out_dtype = compute_dtype(x)

    def fwd(E, x_):
        out, sv = engine.attn_fwd(E, blk, engine.to_nhwc(E, x_))
        return engine.to_nchw(E, out, out_dtype), sv

    def bwd(E, sv, dy):
        dx = engine.attn_bwd(E, blk, sv, engine.to_nhwc(E, dy))
        return (engine.to_nchw(E, dx, torch.float32).to(x.dtype),)

    return block_apply(blk, fwd, bwd, x)


def down_apply(mod, x: torch.Tensor) -> torch.Tensor:
    _require_cuda(x, "Downsample")
    _, out_dtype = compute_dtype(x)

    def fwd(E, x_):
        out, sv = engine.down_fwd(E, mod, engine.to_nhwc(E, x_))
        return engine.to_nchw(E, out, out_dtype), sv

    def bwd(E, sv, dy):
        dx = engine.down_bwd(E, mod, sv, engine.to_nhwc(E, dy), None, False)
        return (engine.to_nchw(E, dx, torch.float32).to(x.dtype),)

    return block_apply(mod, fwd, bwd, x)


def up_apply(mod, x: torch.Tensor) -> torch.Tensor:
    _require_cuda(x, "Upsample")
    _, out_dtype = compute_dtype(x)

    def fwd(E, x_):
        out, sv = engine.up_fwd(E, mod, engine.to_nhwc(E, x_))
        return engine.to_nchw(E, out, out_dtype), sv

    def bwd(E, sv, dy):
        dx = engine.up_bwd(E, mod, sv, engine.to_nhwc(E, dy))
        return (engine.to_nchw(E, dx, torch.float32).to(x.dtype),)

    return block_apply(mod, fwd, bwd, x)


def time_mlp_apply(mlp, t_emb: torch.Tensor) -> torch.Tensor:
    _require_cuda(t_emb, "TimeMLP")

    def fwd(E, e_):
        e32 = e_.float().contiguous()
        temb, sv = engine.time_mlp_fwd(E, mlp, e32)
        return temb, sv

    def bwd(E, sv, dy):
        de = engine.time_mlp_bwd(E, mlp, sv, dy.float().contiguous(), need_dx=True)
        return (de.to(t_emb.dtype),)

    return block_apply(mlp, fwd, bwd, t_emb)


def sinusoid_apply(t: torch.Tensor, dim: int) -> torch.Tensor:
    _require_cuda(t, "SinusoidalPosEmb")
    E = engine.Exec(t.device, _lib.F32, False, False)
    return engine.sinusoid(E, t, dim)
