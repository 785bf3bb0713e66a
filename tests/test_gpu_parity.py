"""GPU parity tests: the CUDA path (through the C ABI / the reference-shaped modules) against the
CPU oracle and the golden fixtures produced by the live reference.

Tolerances (BASELINE.json north_star): fp32 single forward/backward 1e-4 relative; bf16 2e-2
relative; elementwise fp32 kernels 1e-6 absolute (same op order as the reference, no FMA
contraction); samplers: stated per test.
"""
import ctypes as C
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from oracle import ddpm_oracle as O  # noqa: E402  (tests may use the oracle)


def dev():
    return torch.device("cuda", 0)


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


@pytest.fixture(scope="module")
def pkg():
    import ddpm_diffusion_model_b200 as p
    from ddpm_diffusion_model_b200 import _lib, engine
    return p, _lib, engine


# ------------------------------------------------------------------------------------------------
# diffusion elementwise kernels
# ------------------------------------------------------------------------------------------------
def test_elementwise_golden(golden, pkg):
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion, to_image01
    g = golden("elementwise.pt")
    d = Diffusion(T=1000).to(dev())
    cu = lambda k: g[k].to(dev())  # noqa: E731
    x0, eps, noise, ep, t, tp = (cu(k) for k in ("x0", "eps", "noise", "eps_pred", "t", "t_prev"))
    x_t = d.q_sample(x0, t.clone(), eps)
    assert torch.equal(x_t.cpu(), g["q_sample"])
    assert torch.equal(d.q_sample(x0, cu("t_float"), eps).cpu(), g["q_sample_tfloat"])
    fn = lambda a, b: ep  # noqa: E731
    for key, kw in (("ddpm_step", {}), ("ddpm_step_noclamp", {"clamp_x0": False}), ("ddpm_step_dyn", {"dynamic_threshold": 0.995})):
        dd = Diffusion(T=1000, **kw).to(dev())
        out = dd.p_sample_step(fn, x_t, t.clone(), noise=noise)
        assert torch.allclose(out.cpu(), g[key], atol=2e-6, rtol=1e-6), (key, float((out.cpu() - g[key]).abs().max()))
    out = d.p_sample_step_ddim(fn, x_t, t.clone(), tp.clone(), eta=0.0, noise=noise)
    assert torch.allclose(out.cpu(), g["ddim_step_eta0"], atol=2e-6, rtol=1e-6)
    out = d.p_sample_step_ddim(fn, x_t, t.clone(), tp.clone(), eta=0.5, noise=noise)
    assert torch.allclose(out.cpu(), g["ddim_step_eta05"], atol=2e-6, rtol=1e-6)
    dd = Diffusion(T=1000, dynamic_threshold=0.995).to(dev())
    out = dd.p_sample_step_ddim(fn, x_t, t.clone(), tp.clone(), eta=1.0, noise=noise)
    assert torch.allclose(out.cpu(), g["ddim_step_eta1_dyn"], atol=2e-6, rtol=1e-6)
    assert torch.allclose(d.predict_x0(x_t, ep, t.clone()).cpu(), g["predict_x0_clamp"], atol=1e-6)
    assert torch.allclose(dd.predict_x0(x_t, ep, t.clone()).cpu(), g["predict_x0_dyn"], atol=1e-6)
    # loss (fp32 and bf16 eps_pred) + its gradient
    epr = ep.clone().requires_grad_(True)
    loss = d.loss_simple(lambda a, b: epr, x0, t.clone(), noise=eps)
    assert abs(float(loss) - float(g["loss_simple"])) < 2e-6 * max(1, abs(float(g["loss_simple"])))
    loss.backward()
    ref = 2 * (g["eps_pred"] - g["eps"]) / g["eps"].numel()
    assert torch.allclose(epr.grad.cpu(), ref, atol=1e-9, rtol=1e-5)
    lw = d.loss_simple(lambda a, b: ep, x0, t.clone(), noise=eps, weight=cu("weight"))
    assert abs(float(lw) - float(g["loss_simple_weighted"])) < 2e-6 * max(1, abs(float(g["loss_simple_weighted"])))
    eb = ep.to(torch.bfloat16)
    lb = d.loss_simple(lambda a, b: eb, x0, t.clone(), noise=eps)
    tb = O.make_tables()
    assert abs(float(lb) - float(O.loss_simple(tb, lambda a, b: eb.float().cpu(), g["x0"], g["t"], g["eps"]))) < 1e-5
    assert torch.allclose(to_image01(x_t).cpu(), O.to_image01(g["q_sample"]), atol=1e-7)
    # sinusoid
    from ddpm_diffusion_model_b200.model.attention import SinusoidalPosEmb
    assert torch.allclose(SinusoidalPosEmb(64)(t).cpu(), g["sinusoid_64"], atol=2e-4)   # sin/cos of ~1e3 rad
    assert torch.allclose(SinusoidalPosEmb(33)(t).cpu(), g["sinusoid_33"], atol=2e-4)


def test_elementwise_large_properties(pkg):
    """Full-size (B=64 @ 64px) checks through size-independent properties: linearity of q_sample in
    (x0, eps), DDIM eta=0 determinism and noise-independence, t=0 DDPM step ignores noise."""
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    d = Diffusion(T=1000).to(dev())
    torch.manual_seed(0)
    B = 64
    x0 = torch.randn(B, 3, 64, 64, device=dev()); e = torch.randn_like(x0)
    t = torch.randint(0, 1000, (B,), device=dev())
    a = d.q_sample(x0, t, e); b = d.q_sample(2 * x0, t, 2 * e)
    assert torch.allclose(b, 2 * a, atol=1e-5)
    tb = O.make_tables()
    assert torch.allclose(a.cpu(), O.q_sample(tb, x0.cpu(), t.cpu(), e.cpu()), atol=1e-6)
    ep = torch.randn_like(x0)
    tp = (t - 20).clamp(min=0)
    o1 = d.p_sample_step_ddim(lambda x, tt: ep, a, t, tp, eta=0.0, noise=torch.randn_like(a))
    o2 = d.p_sample_step_ddim(lambda x, tt: ep, a, t, tp, eta=0.0, noise=torch.randn_like(a))
    assert torch.equal(o1, o2)
    assert torch.allclose(o1.cpu(), O.ddim_step(tb, ep.cpu(), a.cpu(), t.cpu(), tp.cpu(), torch.zeros_like(a).cpu()), atol=2e-5, rtol=1e-5)
    t0 = torch.zeros(B, dtype=torch.long, device=dev())
    z1 = d.p_sample_step(lambda x, tt: ep, a, t0, noise=torch.randn_like(a))
    z2 = d.p_sample_step(lambda x, tt: ep, a, t0, noise=torch.randn_like(a))
    assert torch.equal(z1, z2)
    # odd sizes exercise the scalar (non-float4) path
    xo = torch.randn(3, 3, 5, 7, device=dev()); eo = torch.randn_like(xo); to = torch.tensor([0, 500, 999], device=dev())
    assert torch.allclose(d.q_sample(xo, to, eo).cpu(), O.q_sample(tb, xo.cpu(), to.cpu(), eo.cpu()), atol=1e-6)


# ------------------------------------------------------------------------------------------------
# primitive kernels against ATen on the CPU (fp32 reference of the same op)
# ------------------------------------------------------------------------------------------------
def _exec(pkg, dt):
    _, _lib, engine = pkg
    return engine.Exec(dev(), dt, True, True)


def _to_act(pkg, E, x):
    _, _lib, engine = pkg
    return engine.to_nhwc(E, x.to(dev()))


def _from_act(pkg, E, a):
    _, _lib, engine = pkg
    return engine.to_nchw(E, a, torch.float32).cpu()


CONV_CASES = [
    # (N, Cin, Cout, H, W, k, stride, pad)
    (2, 3, 32, 16, 16, 3, 1, 1),       # in_conv-like (K=27)
    (2, 32, 3, 16, 16, 3, 1, 1),       # out_conv-like (N=3)
    (2, 64, 64, 8, 8, 3, 1, 1),
    (1, 96, 192, 8, 8, 3, 1, 1),
    (2, 64, 64, 8, 8, 3, 2, 1),        # Downsample
    (2, 96, 64, 8, 8, 1, 1, 0),        # 1x1 skip
    (3, 33, 33, 1, 1, 1, 1, 0),        # odd linear
    (2, 40, 24, 6, 10, 3, 1, 1),       # non-square
]


@pytest.mark.parametrize("dt_name", ["f32", "bf16"])
@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_fwd_dgrad_wgrad(pkg, case, dt_name):
    _, _lib, engine = pkg
    dt = _lib.F32 if dt_name == "f32" else _lib.BF16
    tol = 2e-5 if dt_name == "f32" else 1.5e-2
    N, Ci, Co, H, W, k, s, p = case
    torch.manual_seed(hash(case) % 1000)
    x = torch.randn(N, Ci, H, W)
    w = torch.randn(Co, Ci, k, k) / math.sqrt(Ci * k * k)
    b = torch.randn(Co)
    if dt_name == "bf16":
        x = x.bfloat16().float(); w = w.bfloat16().float()
    xr = x.clone().requires_grad_(True); wr = w.clone().requires_grad_(True)
    y_ref = F.conv2d(xr, wr, b, stride=s, padding=p)
    dy = torch.randn_like(y_ref)
    if dt_name == "bf16":
        dy = dy.bfloat16().float()
    y_ref.backward(dy)

    E = _exec(pkg, dt)
    conv_mod = torch.nn.Conv2d(Ci, Co, k, stride=s, padding=p).to(dev())
    with torch.no_grad():
        conv_mod.weight.copy_(w); conv_mod.bias.copy_(b)
    wf, wd = E.wcache.get(E, conv_mod.weight, dt, True)
    xa = _to_act(pkg, E, x)
    Ho, Wo = y_ref.shape[2:]
    ya = engine.conv(E, xa, wf, E.act(N, Ho, Wo, Co), k, s, p, bias=conv_mod.bias)
    assert rel(_from_act(pkg, E, ya), y_ref) < tol
    # halo must stay zero
    full = ya.buf.t.float()
    assert float(full[:, 0].abs().max()) == 0 and float(full[:, :, 0].abs().max()) == 0
    dya = _to_act(pkg, E, dy)
    mode = _lib.CONV_TRANSPOSED if s > 1 else _lib.CONV_NORMAL
    dxa = engine.conv(E, dya, wd, E.act(N, H, W, Ci), k, s, (k - 1 - p), mode=mode) if s == 1 else \
        engine.conv(E, dya, wd, E.act(N, H, W, Ci), k, s, p, mode=mode)
    assert rel(_from_act(pkg, E, dxa), xr.grad) < tol
    engine.wgrad(E, xa, dya, conv_mod.weight, k, s, p)
    engine.colsum(E, dya, None, conv_mod.bias)
    assert rel(conv_mod.weight.grad, wr.grad) < tol
    assert rel(conv_mod.bias.grad, dy.sum((0, 2, 3))) < tol


def test_conv_epilogues(pkg):
    """bias + per-image time bias + residual + accumulate, channel-slice in/out (concat by layout)."""
    _, _lib, engine = pkg
    E = _exec(pkg, _lib.F32)
    torch.manual_seed(3)
    N, Ci, Co, H, W = 2, 32, 48, 8, 8
    x = torch.randn(N, Ci, H, W); w = torch.randn(Co, Ci, 3, 3) * 0.1; b = torch.randn(Co)
    tb = torch.randn(N, Co); r = torch.randn(N, Co, H, W)
    conv_mod = torch.nn.Conv2d(Ci, Co, 3, padding=1).to(dev())
    with torch.no_grad():
        conv_mod.weight.copy_(w); conv_mod.bias.copy_(b)
    wf, _ = E.wcache.get(E, conv_mod.weight, _lib.F32, False)
    wide_in = E.act(N, H, W, Ci + 16)
    wide_in.buf.t.normal_()                                  # garbage in the other channels + halo
    wide_in.buf.t[:, 0] = 0; wide_in.buf.t[:, -1] = 0; wide_in.buf.t[:, :, 0] = 0; wide_in.buf.t[:, :, -1] = 0
    xin = wide_in.slice(16, Ci)
    xin.interior().copy_(x.permute(0, 2, 3, 1).to(dev()))
    wide_out = E.act(N, H, W, Co + 8)
    out = wide_out.slice(8, Co)
    ra = _to_act(pkg, E, r)
    engine.conv(E, xin, wf, out, 3, 1, 1, bias=conv_mod.bias, tbias=tb.to(dev()), res=ra)
    ref = F.conv2d(x, w, b, padding=1) + tb[:, :, None, None] + r
    assert rel(out.interior().permute(0, 3, 1, 2), ref) < 2e-5
    engine.conv(E, xin, wf, out, 3, 1, 1, accum=True)
    assert rel(out.interior().permute(0, 3, 1, 2), ref + F.conv2d(x, w, None, padding=1)) < 2e-5


def _halo_max(a):
    t = a.buf.t.float()
    return float(max(t[:, 0].abs().max(), t[:, -1].abs().max(), t[:, :, 0].abs().max(), t[:, :, -1].abs().max()))


@pytest.mark.parametrize("dt_name", ["f32", "bf16"])
@pytest.mark.parametrize("shape", [(2, 32, 8, 8), (2, 96, 8, 8), (1, 288, 4, 4), (2, 64, 16, 16), (3, 96, 64, 64),
                                   (2, 192, 16, 16), (2, 192, 32, 32), (2, 96, 12, 20),
                                   (2, 128, 128, 128),        # few large images -> clusters of 16 CTAs
                                   (130, 192, 16, 16), (2, 288, 64, 64), (3, 96, 24, 24), (2, 384, 32, 32), (5, 192, 8, 8),
                                   (2, 32, 4, 4), (7, 384, 16, 16), (4, 512, 16, 16)])
@pytest.mark.parametrize("act", [0, 1])
def test_groupnorm_fwd_bwd(pkg, shape, act, dt_name):
    _, _lib, engine = pkg
    dt = _lib.F32 if dt_name == "f32" else _lib.BF16
    tol = 3e-5 if dt_name == "f32" else 2e-2
    N, Cc, H, W = shape
    torch.manual_seed(Cc + act)
    x = torch.randn(N, Cc, H, W) * 1.7 + 0.3
    dy = torch.randn(N, Cc, H, W)
    if dt_name == "bf16":
        x = x.bfloat16().float(); dy = dy.bfloat16().float()
    gn = torch.nn.GroupNorm(min(32, Cc), Cc, eps=1e-6)
    with torch.no_grad():
        gn.weight.uniform_(0.5, 1.5); gn.bias.normal_()
    xr = x.clone().requires_grad_(True)
    y = gn(xr)
    y = F.silu(y) if act else y
    y.backward(dy)
    gdev = torch.nn.GroupNorm(min(32, Cc), Cc, eps=1e-6).to(dev())
    gdev.load_state_dict(gn.state_dict())
    E = _exec(pkg, dt)
    xa = _to_act(pkg, E, x)
    st = engine.gn_stats(E, xa, gdev.num_groups)
    ya = engine.gn_apply(E, xa, st, gdev, act, 0.0, 0)
    assert rel(_from_act(pkg, E, ya), y) < tol
    # fused stats+apply (one cluster per image) must agree with the two-launch path and the reference (ATen fp32 on the
    # bf16-rounded input: without the activation, the bf16 output is within a rounding step of it)
    yf, stf = engine.gn_fwd(E, xa, gdev, act, 0.0, 0)
    assert rel(_from_act(pkg, E, yf), y) < (6e-3 if dt_name == "bf16" and not act else tol)
    assert torch.allclose(stf, st, rtol=1e-6, atol=1e-6)
    dya = _to_act(pkg, E, dy)
    dxa = engine.gn_bwd(E, xa, st, gdev, act, 0.0, 0, dya, E.act(N, H, W, Cc), False)
    assert rel(_from_act(pkg, E, dxa), xr.grad) < tol
    assert rel(gdev.weight.grad, gn.weight.grad) < tol
    assert rel(gdev.bias.grad, gn.bias.grad) < tol
    # scratch-dy variant with fused column sums (what the UNet backward uses), into a new buffer and in place (dx is dy)
    ctol = 1e-5 if dt_name == "f32" else 2e-3
    for in_place in (False, True):
        gdev.weight.grad = None; gdev.bias.grad = None
        dyb = _to_act(pkg, E, dy)
        cs_nc = torch.full((N, Cc), 7.0, device=dev())
        cbias = torch.nn.Parameter(torch.zeros(Cc, device=dev()))
        dxb = engine.gn_bwd(E, xa, st, gdev, act, 0.0, 0, dyb, dyb if in_place else E.act(N, H, W, Cc), False, colsum_nc=cs_nc,
                            colsum_bias=cbias, dy_scratch=True)
        assert _halo_max(dxb) == 0.0, in_place
        got = _from_act(pkg, E, dxb)
        assert rel(got, xr.grad) < tol, in_place
        assert rel(gdev.weight.grad, gn.weight.grad) < tol, in_place
        assert rel(gdev.bias.grad, gn.bias.grad) < tol, in_place
        # (per-group sums of a GroupNorm gradient are ~0, so compare against the scale of sum|dx|, not of the sum)
        assert float((cs_nc.cpu() - got.sum((2, 3))).abs().max()) < ctol * float(got.abs().sum((2, 3)).max())
        assert float((cbias.grad.cpu() - got.sum((0, 2, 3))).abs().max()) < ctol * float(got.abs().sum((0, 2, 3)).max())
    # accumulate variant: dx += ...
    base = torch.randn(N, Cc, H, W)
    if dt_name == "bf16":
        base = base.bfloat16().float()
    acc = _to_act(pkg, E, base)
    engine.gn_bwd(E, xa, st, gdev, act, 0.0, 0, dya, acc, True)
    assert rel(_from_act(pkg, E, acc), xr.grad + base) < tol
    # no kernel writes the zero halo
    assert max(_halo_max(ya), _halo_max(yf), _halo_max(dxa), _halo_max(acc)) == 0.0


def test_dropout_statistics(pkg):
    """Dropout cannot be bit-matched to ATen's Philox stream (SURVEY §7): check keep rate, scaling,
    determinism for a fixed (seed, step, layer) and that backward uses the same mask."""
    _, _lib, engine = pkg
    from ddpm_diffusion_model_b200 import functional as Fn
    E = _exec(pkg, _lib.F32)
    Fn.seed_dropout(1234, dev())
    E.rng = Fn.rng_state(dev())
    N, Cc, H, W = 4, 64, 16, 16
    x = torch.randn(N, Cc, H, W)
    gn = torch.nn.GroupNorm(32, Cc, eps=1e-6).to(dev())
    xa = _to_act(pkg, E, x)
    st = engine.gn_stats(E, xa, 32)
    y0 = _from_act(pkg, E, engine.gn_apply(E, xa, st, gn, 1, 0.0, 0))
    y1 = _from_act(pkg, E, engine.gn_apply(E, xa, st, gn, 1, 0.25, 7))
    y2 = _from_act(pkg, E, engine.gn_apply(E, xa, st, gn, 1, 0.25, 7))
    y3 = _from_act(pkg, E, engine.gn_apply(E, xa, st, gn, 1, 0.25, 8))
    assert torch.equal(y1, y2) and not torch.equal(y1, y3)
    keep = (y1 != 0) | (y0 == 0)
    rate = float(keep.float().mean())
    assert abs(rate - 0.75) < 0.01, rate
    assert torch.allclose(y1[keep], y0[keep] / 0.75, rtol=1e-5, atol=1e-6)
    dy = torch.ones(N, Cc, H, W)
    dya = _to_act(pkg, E, dy)
    # with gamma=1, beta=0 and act=none the dropped positions contribute nothing to dbeta
    gn2 = torch.nn.GroupNorm(32, Cc, eps=1e-6).to(dev())
    engine.gn_bwd(E, xa, st, gn2, 0, 0.25, 7, dya, E.act(N, H, W, Cc), False)
    yk = _from_act(pkg, E, engine.gn_apply(E, xa, st, gn2, 0, 0.25, 7))
    kept_per_c = ((yk != 0).float().sum((0, 2, 3)) / 0.75)
    assert torch.allclose(gn2.bias.grad.cpu(), kept_per_c, rtol=2e-3, atol=1.0)


@pytest.mark.parametrize("dt_name", ["f32", "bf16"])
@pytest.mark.parametrize("cfg", [(2, 8, 8, 2, 16), (1, 16, 16, 4, 32), (2, 8, 8, 1, 64), (1, 12, 12, 2, 8), (1, 32, 32, 2, 32),
                                 (2, 16, 16, 4, 64), (3, 8, 8, 2, 32)])     # last two: the CelebA256 / low-GPU blocks (tcgen05 forward in bf16)
def test_attention_fwd_bwd(pkg, cfg, dt_name):
    _, _lib, engine = pkg
    dt = _lib.F32 if dt_name == "f32" else _lib.BF16
    tol = 5e-5 if dt_name == "f32" else 2e-2
    B, H, W, heads, d = cfg
    inner = heads * d
    torch.manual_seed(d + heads)
    qkv = torch.randn(B, 3 * inner, H, W)
    do = torch.randn(B, inner, H, W)
    if dt_name == "bf16":
        qkv = qkv.bfloat16().float(); do = do.bfloat16().float()
    qr = qkv.clone().requires_grad_(True)
    N = H * W
    q, k, v = (qr.reshape(B, 3, heads, d, N)[:, i].transpose(-1, -2) for i in range(3))
    o_ref = F.scaled_dot_product_attention(q, k, v).transpose(-1, -2).reshape(B, inner, H, W)
    o_ref.backward(do)
    E = _exec(pkg, dt)
    qa = _to_act(pkg, E, qkv)
    oa = E.act(B, H, W, inner)
    lse = E.f32(B, heads, N)
    _lib.call("ddpm_attn_fwd", C.byref(qa.desc()), C.byref(oa.desc()), heads, d, lse.data_ptr(), dt, E.stream)
    assert rel(_from_act(pkg, E, oa), o_ref) < tol
    doa = _to_act(pkg, E, do)
    dqa = E.act(B, H, W, 3 * inner)
    scratch = E.f32(2, B, heads, N, N)
    _lib.call("ddpm_attn_bwd", C.byref(qa.desc()), C.byref(oa.desc()), C.byref(doa.desc()), lse.data_ptr(),
              C.byref(dqa.desc()), heads, d, scratch.data_ptr(), dt, E.stream)
    assert rel(_from_act(pkg, E, dqa), qr.grad) < tol


def test_upsample_add_colsum(pkg):
    _, _lib, engine = pkg
    E = _exec(pkg, _lib.F32)
    x = torch.randn(2, 24, 4, 6)
    xa = _to_act(pkg, E, x)
    ua = E.act(2, 8, 12, 24)
    _lib.call("ddpm_upsample2x", C.byref(xa.desc()), C.byref(ua.desc()), _lib.F32, E.stream)
    assert torch.equal(_from_act(pkg, E, ua), F.interpolate(x, scale_factor=2, mode="nearest"))
    dy = torch.randn(2, 24, 8, 12)
    dxa = E.act(2, 4, 6, 24)
    _lib.call("ddpm_upsample2x_bwd", C.byref(_to_act(pkg, E, dy).desc()), C.byref(dxa.desc()), _lib.F32, 0, E.stream)
    assert torch.allclose(_from_act(pkg, E, dxa), F.avg_pool2d(dy, 2) * 4, atol=1e-5)
    out_nc = E.f32(2, 24)
    bias = torch.nn.Parameter(torch.zeros(24, device=dev()))
    engine.colsum(E, _to_act(pkg, E, dy), out_nc, bias)
    assert torch.allclose(out_nc.cpu(), dy.sum((2, 3)), atol=1e-4)
    assert torch.allclose(bias.grad.cpu(), dy.sum((0, 2, 3)), atol=1e-4)


# ------------------------------------------------------------------------------------------------
# modules and the whole UNet against golden vectors of the live reference
# ------------------------------------------------------------------------------------------------
def _build(cfg):
    from ddpm_diffusion_model_b200.model.unet_backbone import UNetDenoiser
    kw = dict(cfg)
    kw["attn_resolutions"] = set(kw["attn_resolutions"]); kw["channel_mults"] = tuple(kw["channel_mults"])
    return UNetDenoiser(**kw)


def _unet_case(golden, name, autocast, tol_out, tol_grad, floor=1e-3):
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    g = golden(name)
    sd = g["state_dict"]
    if isinstance(sd, str):
        sd = golden(sd)["state_dict"]
    model = _build(g["cfg"])
    assert [k for k, _ in model.named_parameters()] == g["param_names"]
    model.load_state_dict(sd)
    model = model.to(dev()).train()
    d = Diffusion(T=1000).to(dev())
    x0, t, noise = g["x0"].to(dev()), g["t"].to(dev()), g["noise"].to(dev())
    ctx = torch.autocast("cuda", dtype=torch.bfloat16) if autocast else torch.autocast("cuda", enabled=False)
    with ctx:
        with torch.no_grad():
            eps = model(g["x_t"].to(dev()), t)
        assert eps.dtype == (torch.bfloat16 if autocast else torch.float32)
        assert rel(eps.float(), g["eps_pred"]) < tol_out, rel(eps.float(), g["eps_pred"])
        loss = d.loss_simple(model, x0, t.clone(), noise=noise)
    assert abs(float(loss) - float(g["loss"])) < tol_out * max(1.0, abs(float(g["loss"]))) * 2
    loss.backward()
    gmax = max(float(v.norm()) for v in g["grads"].values())
    worst, worst_k = 0.0, None
    for k, p in model.named_parameters():
        if k not in g["grads"]:
            continue
        ref = g["grads"][k]
        e = float((p.grad.detach().double().cpu() - ref.double()).norm()) / max(float(ref.norm()), floor * gmax)
        if e > worst:
            worst, worst_k = e, k
    assert worst < tol_grad, (worst_k, worst)


def test_unet_fp32_attn(golden):
    _unet_case(golden, "unet_tiny_attn.pt", False, 1e-4, 1e-4)


def test_unet_fp32_noattn_odd_time_dim(golden):
    _unet_case(golden, "unet_tiny_noattn.pt", False, 1e-4, 1e-4)


def test_unet_fp32_other_resolution(golden):
    _unet_case(golden, "unet_tiny_attn_s32.pt", False, 1e-4, 1e-4)


def test_unet_bf16_attn(golden):
    # bf16 tolerance 2e-2 on the forward (north_star); gradients of a random-init net accumulate
    # bf16 rounding through ~20 layers, measured against the fp32 reference: 6e-2 of the tensor norm
    # (tensors whose true gradient is ~0 -- biases in front of a GroupNorm -- are measured against
    # a floor of 1 % of the largest gradient norm)
    _unet_case(golden, "unet_tiny_attn.pt", True, 2e-2, 6e-2, floor=1e-2)


def test_standalone_modules_vs_aten():
    """ResBlock / AttnBlock / Downsample / Upsample / TimeMLP called on their own (the reference's
    testing/test_unet_backbone.py and test_attention.py do this) against the same math in ATen."""
    from ddpm_diffusion_model_b200.model.unet_backbone import ResBlock, Downsample, Upsample
    from ddpm_diffusion_model_b200.model.attention import AttnBlock, TimeMLP
    torch.manual_seed(0)
    blk = ResBlock(64, 128, 64, dropout=0.0).to(dev())
    x = torch.randn(2, 64, 16, 16, device=dev(), requires_grad=True)
    te = torch.randn(2, 64, device=dev(), requires_grad=True)
    y = blk(x, te)
    sd = {"b." + k: v.detach().cpu() for k, v in blk.state_dict().items()}
    xr, ter = x.detach().cpu().requires_grad_(True), te.detach().cpu().requires_grad_(True)
    yr = O.resblock(xr, ter, sd, "b")
    assert rel(y, yr) < 1e-4
    gy = torch.randn_like(y)
    y.backward(gy); yr.backward(gy.cpu())
    assert rel(x.grad, xr.grad) < 1e-4 and rel(te.grad, ter.grad) < 1e-4
    at = AttnBlock(64, num_heads=4, head_dim=16).to(dev())
    xa = torch.randn(2, 64, 8, 8, device=dev(), requires_grad=True)
    ya = at(xa)
    sda = {"a." + k: v.detach().cpu() for k, v in at.state_dict().items()}
    xar = xa.detach().cpu().requires_grad_(True)
    yar = O.attnblock(xar, sda, "a", 4, 16)
    assert rel(ya, yar) < 1e-4
    ya.sum().backward(); yar.sum().backward()
    assert rel(xa.grad, xar.grad) < 1e-4
    dn, up = Downsample(32).to(dev()), Upsample(32).to(dev())
    xd = torch.randn(2, 32, 8, 8, device=dev())
    assert rel(dn(xd), F.conv2d(xd.cpu(), dn.conv.weight.cpu(), dn.conv.bias.cpu(), stride=2, padding=1)) < 1e-4
    assert rel(up(xd), F.conv2d(F.interpolate(xd.cpu(), scale_factor=2), up.conv.weight.cpu(), up.conv.bias.cpu(), padding=1)) < 1e-4
    mlp = TimeMLP(64, 64).to(dev())
    e = torch.randn(3, 64, device=dev())
    ref = F.linear(F.silu(F.linear(e.cpu(), mlp.net[0].weight.cpu(), mlp.net[0].bias.cpu())), mlp.net[2].weight.cpu(), mlp.net[2].bias.cpu())
    assert rel(mlp(e), ref) < 1e-4
    # channels_last input and CPU input behaviour
    xcl = xd.contiguous(memory_format=torch.channels_last)
    assert torch.allclose(dn(xcl), dn(xd), atol=1e-6)
    with pytest.raises(RuntimeError):
        dn.cpu()(xd.cpu())


# ------------------------------------------------------------------------------------------------
# optimiser-side pass, training trajectory, samplers
# ------------------------------------------------------------------------------------------------
def test_param_pass_vs_oracle(pkg):
    _, _lib, engine = pkg
    torch.manual_seed(1)
    n = 10007
    p = torch.randn(n); g = torch.randn(n) * 3; m = torch.randn(n) * 0.1; v = torch.rand(n) * 0.1; e = torch.randn(n)
    scale = 1024.0
    for adamw, wd, clip in ((1, 0.01, 0.5), (0, 0.02, 0.0)):
        npad = (n + 3) // 4 * 4
        pad = lambda z: torch.cat([z, torch.zeros(npad - n)]).to(dev())  # noqa: E731
        P, G, M, V, Em = pad(p), pad(g * scale), pad(m), pad(v), pad(e)
        stats = torch.zeros(4, device=dev()); step = torch.full((1,), 4.0, device=dev())
        sc = torch.full((1,), scale, device=dev())
        st = torch.cuda.current_stream().cuda_stream
        _lib.call("ddpm_param_reduce", G.data_ptr(), npad, stats.data_ptr(), st)
        h = _lib.AdamHyper(1e-3, 0.9, 0.999, 1e-8, wd, clip, 0.99, adamw)
        _lib.call("ddpm_param_update", P.data_ptr(), G.data_ptr(), M.data_ptr(), V.data_ptr(), Em.data_ptr(), npad,
                  stats.data_ptr(), step.data_ptr(), sc.data_ptr(), C.byref(h), st)
        gg, gnorm, inf = O.unscale_and_clip([g * scale], 1.0 / scale, clip if clip > 0 else None)
        assert not inf and abs(float(stats[0]) ** 0.5 / scale - gnorm) < 1e-3 * gnorm
        if adamw:
            pr, mr, vr = O.adamw_step(p, gg[0], m, v, 5, 1e-3, 0.9, 0.999, 1e-8, wd)
        else:
            ref_p = torch.nn.Parameter(p.clone()); ref_p.grad = gg[0].clone()
            opt = torch.optim.Adam([ref_p], lr=1e-3, weight_decay=wd)
            opt.state[ref_p] = {"step": torch.tensor(4.0), "exp_avg": m.clone(), "exp_avg_sq": v.clone()}
            opt.step()
            pr, mr, vr = ref_p.detach(), opt.state[ref_p]["exp_avg"], opt.state[ref_p]["exp_avg_sq"]
        assert torch.allclose(P[:n].cpu(), pr, atol=2e-6, rtol=1e-5)
        assert torch.allclose(M[:n].cpu(), mr, atol=1e-6, rtol=1e-5) and torch.allclose(V[:n].cpu(), vr, atol=1e-6, rtol=1e-5)
        assert torch.allclose(Em[:n].cpu(), O.ema_update(e, pr, 0.99), atol=2e-6, rtol=1e-5)
        assert float(step) == 5.0
    # found-inf: parameters untouched, step not advanced, scaler backs off, EMA still moves
    G[5] = float("inf")
    P0, M0 = P.clone(), M.clone()
    _lib.call("ddpm_param_reduce", G.data_ptr(), npad, stats.data_ptr(), st)
    assert float(stats[1]) == 1.0
    _lib.call("ddpm_param_update", P.data_ptr(), G.data_ptr(), M.data_ptr(), V.data_ptr(), Em.data_ptr(), npad,
              stats.data_ptr(), step.data_ptr(), sc.data_ptr(), C.byref(h), st)
    assert torch.equal(P, P0) and torch.equal(M, M0) and float(step) == 5.0
    tr = torch.zeros(1, dtype=torch.int32, device=dev())
    _lib.call("ddpm_scaler_update", sc.data_ptr(), tr.data_ptr(), stats.data_ptr(), 2.0, 0.5, 3, st)
    assert float(sc) == scale * 0.5 and int(tr) == 0
    stats.zero_()
    for i in range(3):
        _lib.call("ddpm_scaler_update", sc.data_ptr(), tr.data_ptr(), stats.data_ptr(), 2.0, 0.5, 3, st)
    assert float(sc) == scale and int(tr) == 0


def test_train_steps_golden(golden):
    """train_one_epoch (fp32, AdamW + EMA + clip + warm-up) for 3 steps vs the live reference's run."""
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.training_loops.train_one_epoch import train_one_epoch
    from ddpm_diffusion_model_b200.training_loops.ema import EMA
    g = golden("train_steps.pt")
    model = _build(g["cfg"])
    model.load_state_dict(g["init_state_dict"])
    model = model.to(dev())
    d = Diffusion(T=1000, img_size=16).to(dev())
    opt = torch.optim.AdamW(model.parameters(), lr=g["opt"]["lr"], betas=g["opt"]["betas"], weight_decay=g["opt"]["weight_decay"])
    ema = EMA(model, decay=g["ema_decay"])
    # identical t / noise: the reference drew them from the CPU generator; feed them through hooks
    torch.manual_seed(g["rng_seed"])
    draws = []
    for x0 in g["batches"]:
        t = torch.randint(1, 1000, (x0.shape[0],)); draws.append((t, torch.randn_like(x0)))
    it = iter(draws)
    orig_ts, orig_loss = d.sample_timesteps, d.loss_simple
    cur = {}

    def fake_ts(B, device=None):
        cur["t"], cur["n"] = next(it)
        return cur["t"].to(dev())

    def fake_loss(fn, x, t, noise=None, weight=None):
        return orig_loss(fn, x, t, noise=cur["n"].to(dev()), weight=weight)

    d.sample_timesteps, d.loss_simple = fake_ts, fake_loss
    batches = [(b, torch.zeros(b.shape[0])) for b in g["batches"]]
    avg, nb, ni, gs = train_one_epoch(model, d, batches, opt, ema=ema, device="cuda", use_autocast=False,
                                      grad_clip=g["grad_clip"], base_lr=g["base_lr"], warmup_steps=g["warmup_steps"],
                                      global_step=0)
    assert (nb, ni, gs) == (g["n_batches"], g["n_images"], g["global_step"])
    assert abs(avg - g["avg_loss"]) < 1e-4
    tb = O.make_tables()
    spec = O.UNetSpec(**g["cfg"])
    _, _, g0 = O.unet_loss_and_grads(g["init_state_dict"], spec, tb, g["batches"][0], draws[0][0], draws[0][1])
    gmax = max(float(v.norm()) for v in g0.values())
    dead = {k for k, v in g0.items() if float(v.norm()) < 1e-5 * gmax}
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    for k, s in zip(g["param_names"], g["final_ema"]):
        ref, init = g["final_state_dict"][k], g["init_state_dict"][k]
        if k in dead:
            assert float((sd[k] - ref).abs().max()) <= 3 * 2e-3 * 1.01, k
            continue
        moved = float((ref - init).norm())
        assert float((sd[k] - ref).norm()) <= 5e-3 * moved + 1e-6, (k, float((sd[k] - ref).norm()), moved)
    for i, (k, s) in enumerate(zip(g["param_names"], g["final_ema"])):
        if k in dead:
            continue
        init = g["init_state_dict"][k]
        assert float((ema.shadow[i].cpu() - s).norm()) <= 5e-3 * float((s - init).norm()) + 1e-6, k
    # optimizer state is exposed per parameter, like torch's own
    st = opt.state[next(iter(model.parameters()))]
    assert set(st) == {"step", "exp_avg", "exp_avg_sq"} and float(st["step"]) == 3.0


def test_train_bf16_amp_scaler_smoke():
    """bf16 autocast + GradScaler + dropout + grad accumulation: loss decreases, scaler state sane."""
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.model.unet_backbone import UNetDenoiser
    from ddpm_diffusion_model_b200.training_loops.train_one_epoch import train_one_epoch
    from ddpm_diffusion_model_b200.training_loops.grad_scaler import make_grad_scaler
    from ddpm_diffusion_model_b200.training_loops.ema import EMA
    torch.manual_seed(0)
    model = UNetDenoiser(3, 32, (1, 2), 1, {8}, 64, 0.1, 2, 16, 16).to(dev())
    d = Diffusion(T=1000, img_size=16).to(dev())
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3)
    ema = EMA(model, 0.99)
    scaler = make_grad_scaler("cuda", True)
    x = torch.empty(8, 3, 16, 16).uniform_(-1, 1)
    batches = [(x, torch.zeros(8))] * 8
    l0, *_ = train_one_epoch(model, d, batches[:2], opt, scaler=scaler, ema=ema, device="cuda", grad_accum_steps=2)
    for _ in range(6):
        l1, nb, ni, gs = train_one_epoch(model, d, batches, opt, scaler=scaler, ema=ema, device="cuda", grad_accum_steps=2,
                                         use_channels_last=True)
    assert math.isfinite(l1) and l1 < l0, (l0, l1)
    assert float(scaler.get_scale()) == 65536.0 and gs == 4
    assert all(torch.isfinite(p).all() for p in model.parameters())


def test_samplers_golden(golden, tmp_path):
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.testing.ddpim_inference import ddim_infer_sample
    from ddpm_diffusion_model_b200.testing.ddpm_inference import ddpm_infer_sample
    from ddpm_diffusion_model_b200.training_loops.training_utils import ddim_sample
    g = golden("samplers.pt")
    model = _build(g["cfg"]); model.load_state_dict(g["state_dict"]); model = model.to(dev())
    d = Diffusion(T=g["T"], beta_min=g["beta_min"], beta_max=g["beta_max"]).to(dev())
    # identical noise: the reference drew x_T and every randn_like from the CPU generator
    real_randn, real_like = torch.randn, torch.randn_like

    def cpu_randn(*size, device=None, **kw):
        return real_randn(*size, **kw).to(device) if device is not None else real_randn(*size, **kw)

    def cpu_like(x, **kw):
        return real_randn(x.shape).to(x.device)

    torch.randn, torch.randn_like = cpu_randn, cpu_like
    try:
        # fp32 sampler tolerance: max-abs 5e-3 on the [0,1] image (BASELINE.md §4)
        grid = ddim_infer_sample(model, d, n=4, img_size=16, device="cuda", seed=1234, steps=6, eta=0.0, out_path=str(tmp_path / "a.png"))
        assert float((grid.cpu() - g["ddim_grid_eta0"]).abs().max()) < 5e-3
        grid = ddim_infer_sample(model, d, n=3, img_size=16, device="cuda", seed=4321, steps=5, eta=1.0,
                                 schedule_kind="alpha_bar_cosine", out_path=str(tmp_path / "b.png"))
        assert float((grid.cpu() - g["ddim_grid_eta1_abar"]).abs().max()) < 5e-3
        grid = ddpm_infer_sample(model, d, n=4, img_size=16, device="cuda", seed=1234, out_path=str(tmp_path / "c.png"))
        assert float((grid.cpu() - g["ddpm_grid"]).abs().max()) < 5e-3
        x = ddim_sample(model, d, n=4, img_size=16, device="cuda", seed=1234, steps=6, eta=0.0, schedule="karras")
        assert float((x.cpu() - g["ddim_sample_karras"]).abs().max()) < 5e-3
        x = ddim_sample(model, d, n=4, img_size=16, device="cuda", seed=1234, steps=6, eta=0.3, schedule="linear")
        assert float((x.cpu() - g["ddim_sample_linear"]).abs().max()) < 5e-3
    finally:
        torch.randn, torch.randn_like = real_randn, real_like


def test_sampler_cuda_graph_matches_eager(tmp_path, monkeypatch):
    """Opt-in CUDA-graph replay of the sampler step gives bit-identical samples to the eager loop (same seed)."""
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.model.unet_backbone import UNetDenoiser
    from ddpm_diffusion_model_b200.testing.ddpim_inference import ddim_infer_sample
    torch.manual_seed(0)
    model = UNetDenoiser(3, 32, (1, 2), 1, {8}, 64, 0.0, 2, 16, 16).to(dev()).eval()
    d = Diffusion(T=200).to(dev())
    outs = []
    for flag in ("0", "1"):
        monkeypatch.setenv("DDPM_B200_GRAPHS", flag)
        outs.append(ddim_infer_sample(model, d, n=4, img_size=16, device="cuda", seed=7, steps=8, eta=0.5, out_path=str(tmp_path / f"g{flag}.png")))
    assert torch.equal(outs[0], outs[1])


def test_low_gpu_model_fp32_vs_oracle():
    """The BASELINE config-1 model (low-GPU UNet, 12.68 M params) at B=2: forward vs the CPU oracle."""
    from ddpm_diffusion_model_b200.model.unet_backbone import build_unet_64x64
    torch.manual_seed(0)
    kw = dict(base_channels=96, channel_mults=(1, 2, 2, 2), num_res_blocks=1, attn_resolutions={8}, num_heads=2, head_dim=32, dropout=0.1)
    model = build_unet_64x64(**kw).to(dev()).eval()
    assert sum(p.numel() for p in model.parameters()) == 12680259
    x = torch.empty(2, 3, 64, 64, device=dev()).uniform_(-1, 1)
    t = torch.tensor([10, 900], device=dev())
    with torch.no_grad():
        y = model(x, t)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            yb = model(x, t)
    spec = O.UNetSpec(in_channels=3, time_embed_dim=512, img_resolution=64, **kw)
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    with torch.no_grad():
        yr = O.unet_forward(sd, spec, x.cpu(), t.cpu())
    assert rel(y, yr) < 1e-4, rel(y, yr)
    assert rel(yb.float(), yr) < 2e-2, rel(yb.float(), yr)


def test_bf16_training_trajectory_tracks_the_fp32_oracle():
    """End to end: 25 optimiser steps of the bf16 tensor-core path (autocast + GradScaler + fused AdamW/EMA/clip through
    train_one_epoch) against the fp32 oracle stepping the same weights on the same images, timesteps and noise (the
    oracle is plain torch and runs on the GPU here so the test takes seconds).  bf16 cannot match step for step to
    1e-4, so the bar is on the trajectory: every loss within 3 %, and final weights / EMA within 20 % of the distance
    travelled (Adam's normalised update turns bf16 noise on the small gradients into O(lr) differences per step;
    measured 12 %)."""
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.training_loops.ema import EMA
    from ddpm_diffusion_model_b200.training_loops.grad_scaler import make_grad_scaler
    from ddpm_diffusion_model_b200.training_loops.train_one_epoch import train_one_epoch
    cfg = dict(in_channels=3, base_channels=32, channel_mults=(1, 2, 2), num_res_blocks=1, attn_resolutions={8},
               time_embed_dim=128, dropout=0.0, num_heads=2, head_dim=16, img_resolution=32)
    torch.manual_seed(0)
    model = _build(cfg).to(dev()).train()
    init = {k: v.detach().clone() for k, v in model.state_dict().items()}
    d = Diffusion(T=1000, img_size=32).to(dev())
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3, betas=(0.9, 0.999), weight_decay=0.0)
    ema = EMA(model, decay=0.9)
    steps, B = 25, 16
    gen = torch.Generator().manual_seed(42)
    data = [(torch.empty(B, 3, 32, 32).uniform_(-1, 1, generator=gen), torch.randint(1, 1000, (B,), generator=gen),
             torch.randn(B, 3, 32, 32, generator=gen)) for _ in range(steps)]
    it = iter(data)
    cur = {}
    orig_loss = d.loss_simple
    d.sample_timesteps = lambda Bn, device=None: cur.__setitem__("k", next(it)) or cur["k"][1].to(dev())
    d.loss_simple = lambda fn, x, t, noise=None, weight=None: orig_loss(fn, x, t, noise=cur["k"][2].to(dev()), weight=weight)
    losses = []
    scaler = make_grad_scaler("cuda", True)
    for x0, _, _ in data:
        avg, *_ = train_one_epoch(model, d, [(x0, torch.zeros(B))], opt, scaler=scaler, ema=ema, device="cuda", grad_clip=1.0)
        losses.append(avg)
    # ---- oracle, fp32, same everything
    spec, tb = O.UNetSpec(**cfg), {k: v.to(dev()) for k, v in O.make_tables().items()}
    sd = {k: v.clone() for k, v in init.items()}
    o_opt, o_ema, o_losses = {}, {k: v.clone() for k, v in init.items()}, []
    for i, (x0, t, n) in enumerate(data):
        loss, _, sd, o_opt, o_ema = O.train_step(sd, spec, tb, x0.to(dev()), t.to(dev()), n.to(dev()), o_opt, o_ema, lr=1e-3,
                                                 step=i + 1, grad_clip=1.0, ema_decay=0.9)
        o_losses.append(float(loss))
    worst = max(abs(a - b) / b for a, b in zip(losses, o_losses))
    assert worst < 3e-2, (worst, losses[-3:], o_losses[-3:])
    assert o_losses[-1] < 0.8 * o_losses[0]                       # it actually trains
    num = sum(float((model.state_dict()[k].float() - sd[k]).norm()) ** 2 for k in sd) ** 0.5
    den = sum(float((sd[k] - init[k]).norm()) ** 2 for k in sd) ** 0.5
    assert num < 0.2 * den, (num, den)
    e_num = sum(float((s.float() - o_ema[k]).norm()) ** 2 for s, k in zip(ema.shadow, sd)) ** 0.5
    assert e_num < 0.2 * den, (e_num, den)


def test_batched_weight_repack_matches_the_per_weight_kernel():
    """WeightCache.repack_all (one tile-transposing launch for every packed copy, after the optimiser step) against
    ddpm_pack_weights per weight: odd channel counts, channel padding, 3x3 / 1x1 / linear, fp32 and bf16 copies."""
    from ddpm_diffusion_model_b200 import _lib, engine
    dev = torch.device("cuda", 0)
    torch.manual_seed(5)
    shapes = [((96, 3, 3, 3), 16, 0), ((192, 96, 3, 3), 0, 0), ((96, 288, 1, 1), 0, 0), ((100, 70, 3, 3), 80, 112),
              ((384, 96), 0, 0), ((3, 96, 3, 3), 0, 16), ((33, 17, 1, 1), 32, 48)]
    for dt in (_lib.BF16, _lib.F32):
        cache = engine.WeightCache()
        E = engine.Exec(dev, dt, True, True, wcache=cache)
        ws = [torch.nn.Parameter(torch.randn(*s, device=dev)) for s, _, _ in shapes]
        for w, (_, cip, cop) in zip(ws, shapes):
            cache.get(E, w, dt, True, cip, cop)
        with torch.no_grad():
            for w in ws:
                w.mul_(0.5).add_(0.25)                     # what an optimiser step does (same storage, new values)
        assert cache.repack_all(E.stream)
        got = [(cache.entries[(id(w), dt, cip, cop)][1].clone(), cache.entries[(id(w), dt, cip, cop)][2].clone())
               for w, (_, cip, cop) in zip(ws, shapes)]
        fresh = engine.WeightCache()
        for w, (_, cip, cop), (gf, gd) in zip(ws, shapes, got):
            rf, rd = fresh.get(E, w, dt, True, cip, cop)
            torch.cuda.synchronize()
            assert torch.equal(gf, rf) and torch.equal(gd, rd), (tuple(w.shape), cip, cop, dt)
