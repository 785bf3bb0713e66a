"""IEEE half (DDPM_F16) end to end: the tensor-core convolution, weight gradient and attention against float64, GroupNorm +
SiLU + dropout against float64, IEEE overflow, the dtype rule of the C ABI, the UNet under torch.autocast("cuda") against
the fp32 oracle, the samplers, and a user AMP loop with torch's GradScaler.

The case lists, planner transcriptions, fp64 criteria and the dropout-mask emulator are imported from the bf16 test modules
(helpers only, so pytest does not collect their tests twice).  fp16 has 11 significant bits: unit round-off u = 2^-11.
"""
import ctypes as C
import math
import os
import tempfile

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import test_gpu_conv_fp64 as CV
from test_gpu_conv_fp64 import (CONV_CASES, WGRAD_CASES, case_plan, conv_units, halo_zero, judge, launched_kernels,
                                      nchw64, plan_str, spot_check_conv, wcase_plan, wgrad_units, with_mode)
from test_gpu_gn_dropout import (EPS, STEP, dropout_key, group_sums, keep_mask, keep_scale, reference, thr16)

U_F16 = 2.0 ** -11
DDPM_E_ARG = -1


def dev():
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def mods():
    from ddpm_diffusion_model_b200 import _lib, engine
    yield _lib, engine
    _lib.lib.ddpm_set_tc_mode(1, 0)
    _lib.lib.ddpm_set_force_simt(0)


def judge_f16(*args, **kw):
    """test_gpu_conv_fp64.judge with fp16's unit round-off in place of bf16's (criteria 1 and 2 for 16-bit outputs)."""
    saved = CV.U_BF16, CV.RMS_BF16
    CV.U_BF16 = CV.RMS_BF16 = U_F16
    try:
        return judge(*args, **kw)
    finally:
        CV.U_BF16, CV.RMS_BF16 = saved


# ================================================================================================================
# CPU
# ================================================================================================================
def test_f16_code_matches_the_header():
    from ddpm_diffusion_model_b200 import _lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "include", "ddpm_b200.h")) as f:
        hdr = f.read()
    import re
    m = re.search(r"#define DDPM_F16 (\d+)", hdr)
    assert m and int(m.group(1)) == _lib.F16 == 2
    assert (_lib.F32, _lib.BF16) == (0, 1)


def _silu_exact(z):
    return z / (1.0 + np.exp(-z))


def _silu_tanh_worst(z):
    # the bf16 kernels' form: h = z/2, silu = h + h*tanh(h) with tanh.approx's relative error of 2^-11, at its worst sign
    h = z / 2.0
    t = np.tanh(h)
    return h + h * t * (1.0 - np.sign(h * t) * 2.0 ** -11)


def fp16_silu_bound(ref, z):
    """Per-element bound of the fp16 GroupNorm forward: two fp16 ulps of the result plus a floor for the fp32 affine."""
    return 2.0 * U_F16 * np.abs(ref) + 2e-6 * (np.abs(z) + 1.0)


def test_exact_silu_meets_the_fp16_bound_and_the_tanh_form_does_not():
    z = np.linspace(-8.0, 8.0, 20001)
    ref = _silu_exact(z)
    exact16 = _silu_exact(z.astype(np.float32)).astype(np.float16).astype(np.float64)
    tanh16 = _silu_tanh_worst(z.astype(np.float32)).astype(np.float16).astype(np.float64)
    bound = fp16_silu_bound(ref, z)
    assert (np.abs(exact16 - ref) <= bound).all()
    bad = np.abs(tanh16 - ref) > bound
    assert bad.any()
    # where SiLU cancels the tanh form is off by many fp16 ulps (about 5 at z = -3, about 200 at z = -6)
    for zz, ulps in ((-3.0, 3), (-6.0, 50)):
        i = int(np.argmin(np.abs(z - zz)))
        ulp = np.spacing(np.float16(ref[i])).astype(np.float64)
        assert abs(_silu_tanh_worst(np.float32(zz)) - ref[i]) > ulps * ulp


# ================================================================================================================
# GPU: convolution and weight gradient against fp64, tile by tile
# ================================================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("case", CONV_CASES, ids=[c["name"] for c in CONV_CASES])
def test_conv_fp16_fp64(mods, case):
    _lib, engine = mods
    c = case
    torch.manual_seed(11)
    N, Ci, Co, H, W, k = c["N"], c["cin"], c["cout"], c["H"], c["W"], c["k"]
    dgrad = c["op"] == "dgrad"
    E = engine.Exec(dev(), _lib.F16, False, False)
    wshape = (Ci, Co, k, k) if dgrad else (Co, Ci, k, k)
    w = torch.nn.Parameter(torch.randn(*wshape, device=dev()) / math.sqrt(wshape[1] * k * k))
    wf, wd = E.wcache.get(E, w, _lib.F16, dgrad)
    wh = w.detach().half()
    wk = wh.flip(2, 3).transpose(0, 1).contiguous() if dgrad else wh
    wpack = wd if dgrad else wf
    assert wpack.dtype == torch.float16
    assert torch.equal(wpack.view(Co, k * k, Ci), wk.permute(0, 2, 3, 1).reshape(Co, k * k, Ci))
    w64 = wk.double()
    x = E.act(N, H, W, Ci)
    x.interior().normal_()
    bias = torch.randn(Co, device=dev()) if c["bias"] else None
    tb = torch.randn(N, Co, device=dev()) if c["tbias"] else None
    res = None
    if c["res"]:
        res = E.act(N, H, W, Co)
        res.interior().normal_()
    in2 = w2pack = w2 = None
    if c["c2"]:
        wide_in = E.act(N, H, W, c["c2"] + 32)
        wide_in.interior().normal_()
        in2 = wide_in.slice(16, c["c2"])
        w2 = torch.nn.Parameter(torch.randn(Co, c["c2"], 1, 1, device=dev()) / math.sqrt(c["c2"]))
        w2pack, _ = E.wcache.get(E, w2, _lib.F16, False)
    if c["out_slice"] is not None:
        c0, wide = c["out_slice"]
        wide_out = E.act(N, H, W, wide)
        out = wide_out.slice(c0, Co)
    else:
        wide_out = E.act(N, H, W, Co)
        out = wide_out
    wide_out.interior().fill_(3.0)
    if c["accum"]:
        out.interior().normal_()
    elif c["out_slice"] is None:
        out.interior().fill_(float("nan"))
    acc0 = nchw64(out).clone() if c["accum"] else None
    before = wide_out.buf.t.clone()

    plan = case_plan(c)                        # fp16 plans exactly as bf16: same element size, same shared memory
    run = lambda: engine.conv(E, x, wpack, out, k, 1, k // 2, bias=bias, tbias=tb, res=res, accum=c["accum"],  # noqa: E731
                              in2=in2, w2pack=w2pack)
    ks = with_mode(_lib, c["flags"], lambda: launched_kernels(run))
    assert len(ks) == 1 and plan["kernel"].replace("conv_tc2_kernel", "conv_tc2_f16_kernel") in ks[0][0], (ks, plan_str(plan))
    assert ks[0][1][0] == plan["grid"], (ks, plan_str(plan))
    after = wide_out.buf.t
    assert halo_zero(after), "the kernel wrote the zero halo"
    if c["out_slice"] is not None:
        keep = torch.ones(wide, dtype=torch.bool, device=dev())
        keep[c0:c0 + Co] = False
        assert torch.equal(after[..., keep].view(torch.int16), before[..., keep].view(torch.int16))

    x64 = nchw64(x)
    ref = F.conv2d(x64, w64, padding=k // 2)
    A = F.conv2d(x64.abs(), w64.abs(), padding=k // 2)
    K = k * k * Ci
    extra = torch.zeros_like(ref)
    if in2 is not None:
        x2 = nchw64(in2)
        w264 = w2.detach().half().double()
        extra = extra + F.conv2d(x2, w264)
        A += F.conv2d(x2.abs(), w264.abs())
        K += c["c2"]
    for t4 in ([bias.double()[None, :, None, None]] if bias is not None else []) + \
              ([tb.double()[:, :, None, None]] if tb is not None else []) + \
              ([nchw64(res)] if res is not None else []) + ([acc0] if acc0 is not None else []):
        extra = extra + t4
        A += t4.abs()
        K += 1
    spot_check_conv(x64, w64, ref, 1, k // 2)
    ref = ref + extra
    unit = conv_units(N, H, W, Co, plan["NT"], device=dev())
    ok, c1, c2, wu, det = judge_f16(nchw64(out), ref, A, K, unit, int(unit.max()) + 1, True)
    print(f"\nMARGIN fp16 conv | {c['name']} | c1 {c1:.3f} | c2 {c2:.3f} | {plan_str(plan)}")
    assert ok, (c["name"], plan_str(plan), det)


@pytest.mark.gpu
@pytest.mark.parametrize("case", WGRAD_CASES, ids=[c["name"] for c in WGRAD_CASES])
def test_wgrad_fp16_fp64(mods, case):
    _lib, engine = mods
    c = case
    torch.manual_seed(12)
    N, Ci, Co, H, W, k = c["N"], c["cin"], c["cout"], c["H"], c["W"], c["k"]
    E = engine.Exec(dev(), _lib.F16, True, True)
    x = E.act(N, H, W, Ci)
    x.interior().normal_()
    dy = E.act(N, H, W, Co)
    dy.interior().normal_()
    ci_v, co_v = c["cin_valid"] or Ci, c["cout_valid"] or Co
    w = torch.nn.Parameter(torch.zeros(co_v, ci_v, k, k, device=dev()))
    b = torch.nn.Parameter(torch.zeros(co_v, device=dev()))
    w.grad = torch.randn_like(w) * 0.1
    b.grad = torch.randn_like(b)
    g0, gb0 = w.grad.double().clone(), b.grad.double().clone()
    plan = wcase_plan(c)
    run = lambda: engine.wgrad(E, x, dy, w, k, 1, k // 2, bias=b if c["bias"] else None)  # noqa: E731
    ks = with_mode(_lib, c["flags"], lambda: launched_kernels(run))
    names = [n for n, _ in ks]
    assert len(ks) == 2 and plan["kernel"].replace("_kernel", "_f16_kernel(") in names[0] and "wgrad_reduce_kernel" in names[1], (names, plan_str(plan))
    assert ks[0][1] == plan["grid"], (ks, plan_str(plan))
    x64, dy64 = nchw64(x), nchw64(dy)
    ref = torch.nn.grad.conv2d_weight(x64, (Co, Ci, k, k), dy64, padding=k // 2)
    A = torch.nn.grad.conv2d_weight(x64.abs(), (Co, Ci, k, k), dy64.abs(), padding=k // 2)[:co_v, :ci_v] + g0.abs()
    ref = ref[:co_v, :ci_v] + g0
    unit = wgrad_units(co_v, ci_v, k, plan["NT"], device=dev())
    ok, c1, c2, wu, det = judge_f16(w.grad, ref, A, N * H * W + plan["splits"] + 1, unit, int(unit.max()) + 1, False)
    assert ok, (c["name"], plan_str(plan), det)
    if c["bias"]:
        refb = dy64.sum((0, 2, 3))[:co_v] + gb0
        Ab = dy64.abs().sum((0, 2, 3))[:co_v] + gb0.abs()
        Kb = N * H * W + plan["splits"] * plan["ngrp"] + 1
        ok, c1, c2, wu, det = judge_f16(b.grad, refb, Ab, Kb, torch.arange(co_v, device=dev()), co_v, False)
        assert ok, (c["name"], "dbias", plan_str(plan), det)


@pytest.mark.gpu
@pytest.mark.parametrize("stride_path", ["down_fwd", "down_bwd", "up_fwd", "up_bwd"])
def test_resampling_blocks_fp16_vs_fp64(mods, stride_path):
    """Stride-2 down, zero-interleaved down_bwd, the four folded up-sampling phases and up_bwd, through the stand-alone
    modules in fp16 against their float64 math on the same fp16-rounded operands."""
    from ddpm_diffusion_model_b200.model.unet_backbone import Downsample, Upsample
    torch.manual_seed(5)
    ch, N, H = 64, 4, 16
    mod = (Downsample(ch) if stride_path.startswith("down") else Upsample(ch)).to(dev())
    with torch.no_grad():
        mod.conv.weight.copy_(mod.conv.weight.half().float())
        mod.conv.bias.normal_()
    x = torch.randn(N, ch, H, H, device=dev()).half()
    w64, b64 = mod.conv.weight.double(), mod.conv.bias.double()

    def ref_f(xx):
        if stride_path.startswith("down"):
            return F.conv2d(xx, w64, b64, stride=2, padding=1)
        return F.conv2d(F.interpolate(xx, scale_factor=2, mode="nearest"), w64, b64, padding=1)

    if stride_path.endswith("fwd"):
        with torch.no_grad():
            y = mod(x)
        assert y.dtype == torch.float16
        ref = ref_f(x.double())
        nrel = float((y.double() - ref).norm() / ref.norm())
        assert nrel < 2e-3, nrel
    else:
        xr = x.clone().requires_grad_(True)
        y = mod(xr)
        g = torch.randn_like(y)
        y.backward(g)
        assert xr.grad.dtype == torch.float16
        x64 = x.double().requires_grad_(True)
        ref_f(x64).backward(g.double())
        nrel = float((xr.grad.double() - x64.grad).norm() / x64.grad.norm())
        assert nrel < 3e-3, nrel


# ================================================================================================================
# GPU: IEEE overflow
# ================================================================================================================
@pytest.mark.gpu
def test_conv_overflow_is_ieee_inf(mods):
    _lib, engine = mods
    E = engine.Exec(dev(), _lib.F16, False, False)
    N, Ci, Co, H = 2, 64, 64, 16
    x = E.act(N, H, H, Ci)
    x.interior().uniform_(0.5, 1.0)
    w = torch.nn.Parameter(torch.full((Co, Ci, 1, 1), 0.0, device=dev()))
    with torch.no_grad():
        w[: Co // 2] = 1500.0          # 64 channels x 0.5..1.0 x 1500 > 65520: +inf
        w[Co // 2: Co // 2 + 8] = -1500.0
        w[Co // 2 + 8:] = 1.0
    wf, _ = E.wcache.get(E, w, _lib.F16, False)
    out = E.act(N, H, H, Co)
    engine.conv(E, x, wf, out, 1, 1, 0)
    torch.cuda.synchronize()
    y = out.interior().float()
    ref = nchw64(x).permute(0, 2, 3, 1) @ w.detach().double()[:, :, 0, 0].t()
    big = ref.abs() > 65520
    assert bool(big[..., : Co // 2 + 8].all()) and not bool(big[..., Co // 2 + 8:].any())
    assert bool((y[big] == torch.sign(ref[big]).float() * math.inf).all())
    assert bool(torch.isfinite(y[~big]).all())


@pytest.mark.gpu
def test_mse_bwd_overflow_writes_inf(mods):
    _lib, _ = mods
    B, chw = 4, 3 * 16 * 16
    pred = torch.randn(B, chw, device=dev()).half()
    noise = torch.randn(B, chw, device=dev())
    gout = torch.tensor([2.0 ** 40], device=dev())
    dpred = torch.zeros_like(pred)
    rc = _lib.lib.ddpm_mse_bwd(C.c_void_p(pred.data_ptr()), _lib.F16, C.c_void_p(noise.data_ptr()), None,
                               C.c_void_p(gout.data_ptr()), C.c_void_p(dpred.data_ptr()), B, chw,
                               C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0
    torch.cuda.synchronize()
    ref = 2.0 * (pred.double() - noise.double()) * 2.0 ** 40 / (B * chw)
    big, small = ref.abs() > 65600, ref.abs() < 65400
    assert bool(big.any()) and bool((dpred[big].double() == torch.sign(ref[big]) * math.inf).all())
    assert bool(torch.isfinite(dpred[small]).all())


# ================================================================================================================
# GPU: GroupNorm + SiLU + dropout in fp16 against fp64
# ================================================================================================================
def _gn_view(engine, _lib, N, Cc, H, W, halo, misaligned):
    off, extra = (1, 3) if misaligned else (0, 0)
    t = torch.zeros(N, H + 2 * halo, W + 2 * halo, Cc + extra, dtype=torch.float16, device=dev())
    return engine.Act.wrap(t, N, H, W, Cc + extra, _lib.F16, halo).slice(off, Cc)


def _put(a, x):
    a.interior().copy_(x.permute(0, 2, 3, 1).to(a.buf.t.dtype))


def _get(a):
    return a.interior().permute(0, 3, 1, 2).double()


def _s():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


@pytest.mark.gpu
@pytest.mark.parametrize("p", [0.0, 0.1])
@pytest.mark.parametrize("halo", [0, 1])
@pytest.mark.parametrize("path", ["vector", "scalar"])
def test_groupnorm_silu_dropout_fp16_fp64(mods, path, halo, p):
    _lib, engine = mods
    L = _lib.lib
    N, Cc, H, W, G, layer, seed = 2, 96, 8, 12, 32, 3, 1234
    gen = torch.Generator(device=dev()).manual_seed(7)
    x = (torch.randn(N, Cc, H, W, generator=gen, device=dev(), dtype=torch.float64) * 2).half().double()
    dy = torch.randn(N, Cc, H, W, generator=gen, device=dev(), dtype=torch.float64).half().double()
    gamma = (0.5 + torch.rand(Cc, generator=gen, device=dev(), dtype=torch.float64)).float()
    beta = torch.randn(Cc, generator=gen, device=dev(), dtype=torch.float64).float()
    rng = torch.tensor([seed, STEP], dtype=torch.int64, device=dev())
    keep = keep_mask(N, H, W, Cc, dropout_key(seed, STEP, layer), thr16(p)).to(dev()) if p > 0 else None
    sc = keep_scale(p) if p > 0 else 1.0
    ref = reference(x, gamma, beta, G, 1, keep, sc, dy)
    mis = path == "scalar"
    xv, ov = _gn_view(engine, _lib, N, Cc, H, W, halo, mis), _gn_view(engine, _lib, N, Cc, H, W, halo, mis)
    _put(xv, x)
    stats = torch.zeros(N, G, 2, dtype=torch.float64, device=dev())
    rc = L.ddpm_gn_fwd(C.byref(xv.desc()), _lib.F16, G, C.c_void_p(stats.data_ptr()), C.c_void_p(gamma.data_ptr()),
                       C.c_void_p(beta.data_ptr()), C.c_float(EPS), 1, C.c_float(p),
                       C.c_void_p(rng.data_ptr()) if p > 0 else None, layer, C.byref(ov.desc()), _s())
    assert rc == 0
    torch.cuda.synchronize()
    rs = group_sums(x, G)
    assert float(((stats - rs).abs() / (rs.abs() + 1)).max()) < 1e-6
    y = _get(ov)
    bound = torch.from_numpy(fp16_silu_bound(ref["y"].cpu().numpy(), ref["z"].cpu().numpy() * sc)).to(dev())
    bad = (y - ref["y"]).abs() > bound
    assert not bool(bad.any()), f"{int(bad.sum())} forward elements outside 2 fp16 ulps + floor"

    dyv, dxv = _gn_view(engine, _lib, N, Cc, H, W, halo, mis), _gn_view(engine, _lib, N, Cc, H, W, halo, mis)
    _put(dyv, dy)
    dgamma, dbeta = torch.zeros(Cc, device=dev()), torch.zeros(Cc, device=dev())
    cs_nc, cs_c = torch.zeros(N, Cc, device=dev()), torch.zeros(Cc, device=dev())
    rc = L.ddpm_gn_bwd_colsum(C.byref(xv.desc()), _lib.F16, G, C.c_void_p(stats.data_ptr()), C.c_void_p(gamma.data_ptr()),
                              C.c_void_p(beta.data_ptr()), C.c_float(EPS), 1, C.c_float(p),
                              C.c_void_p(rng.data_ptr()) if p > 0 else None, layer, C.byref(dyv.desc()),
                              C.byref(dxv.desc()), 0, C.c_void_p(dgamma.data_ptr()), C.c_void_p(dbeta.data_ptr()),
                              C.c_void_p(cs_nc.data_ptr()), C.c_void_p(cs_c.data_ptr()), 0, _s())
    assert rc == 0
    torch.cuda.synchronize()
    dx = _get(dxv)
    dmax = float(ref["dx"].abs().max())
    assert float((dx - ref["dx"]).abs().max()) <= 4 * U_F16 * dmax
    for name, got, want in (("dgamma", dgamma, ref["dgamma"]), ("dbeta", dbeta, ref["dbeta"])):
        nrel = float((got.double() - want).norm() / want.norm())
        assert nrel < 1e-3, (name, nrel)
    tot = dx.abs().sum((2, 3)).max()
    assert float((cs_nc.double() - dx.sum((2, 3))).abs().max()) <= 1e-4 * float(tot)
    assert float((cs_c.double() - dx.sum((0, 2, 3))).abs().max()) <= 1e-4 * float(tot) * N


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["vector", "scalar"])
def test_dropout_mask_readout_fp16_equals_bf16(mods, path):
    """gamma = 0, beta = 1, no activation: the output is keep_scale where kept and 0 where dropped, bit for bit the
    documented mask, and the same elements as the bf16 kernels drop for the same (seed, step, layer)."""
    _lib, engine = mods
    L = _lib.lib
    N, Cc, H, W, G, p, seed, layer = 2, 96, 6, 10, 32, 0.1, 1234, 5
    keep = keep_mask(N, H, W, Cc, dropout_key(seed, STEP, layer), thr16(p)).to(dev())
    outs = {}
    for dt, tdt in ((_lib.F16, torch.float16), (_lib.BF16, torch.bfloat16)):
        off, extra = (1, 3) if path == "scalar" else (0, 0)
        mk = lambda: engine.Act.wrap(torch.zeros(N, H + 2, W + 2, Cc + extra, dtype=tdt, device=dev()),  # noqa: E731
                                     N, H, W, Cc + extra, dt, 1).slice(off, Cc)
        xv, ov = mk(), mk()
        _put(xv, torch.randn(N, Cc, H, W, device=dev()))
        stats = group_sums(_get(xv), G).contiguous()
        gamma, beta = torch.zeros(Cc, device=dev()), torch.ones(Cc, device=dev())
        rng = torch.tensor([seed, STEP], dtype=torch.int64, device=dev())
        rc = L.ddpm_gn_apply(C.byref(xv.desc()), dt, G, C.c_void_p(stats.data_ptr()), C.c_void_p(gamma.data_ptr()),
                             C.c_void_p(beta.data_ptr()), C.c_float(EPS), 0, C.c_float(p), C.c_void_p(rng.data_ptr()),
                             layer, C.byref(ov.desc()), _s())
        assert rc == 0
        torch.cuda.synchronize()
        outs[dt] = _get(ov)
    y = outs[_lib.F16]
    assert torch.equal(y != 0, keep)
    assert bool((y[keep] == torch.tensor(keep_scale(p), dtype=torch.float16).double().item()).all())
    assert torch.equal(y != 0, outs[_lib.BF16] != 0)


# ================================================================================================================
# GPU: attention on tcgen05 in fp16 against fp64
# ================================================================================================================
def _attn_ref(q, k, v, scale):
    s = torch.einsum("bhid,bhjd->bhij", q, k) * scale
    return torch.softmax(s, -1) @ v, torch.logsumexp(s, -1)


ATTN_SHAPES = [(2, 2, 32, 8, 8), (1, 2, 64, 16, 16), (1, 1, 64, 24, 20), (1, 1, 128, 16, 16), (2, 1, 48, 8, 8)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ATTN_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_attention_fp16_fp64(mods, shape):
    _lib, engine = mods
    L = _lib.lib
    B, heads, d, H, W = shape
    tc = d in (32, 64, 128)
    E = engine.Exec(dev(), _lib.F16, False, False)
    N, inner = H * W, heads * d
    qkv, out, dout, dqkv = E.act(B, H, W, 3 * inner), E.act(B, H, W, inner), E.act(B, H, W, inner), E.act(B, H, W, 3 * inner)
    torch.manual_seed(3)
    qkv.interior().normal_()
    dout.interior().normal_()
    lse = torch.empty(B, heads, N, device=dev())
    scr = torch.empty(int(L.ddpm_attn_bwd_scratch_floats(C.byref(qkv.desc()), C.byref(out.desc()), heads, d, _lib.F16)),
                      device=dev())

    def run():
        assert L.ddpm_attn_fwd(C.byref(qkv.desc()), C.byref(out.desc()), heads, d, C.c_void_p(lse.data_ptr()), _lib.F16, _s()) == 0
        assert L.ddpm_attn_bwd(C.byref(qkv.desc()), C.byref(out.desc()), C.byref(dout.desc()), C.c_void_p(lse.data_ptr()),
                               C.byref(dqkv.desc()), heads, d, C.c_void_p(scr.data_ptr()), _lib.F16, _s()) == 0
    names = [n for n, _ in launched_kernels(run)]
    if tc:
        for kname in ("attn_fwd_tc_kernel", "attn_bwd_dq_tc_kernel", "attn_bwd_dkv_tc_kernel"):
            assert any(kname in n and "__half" in n for n in names), names
    else:
        assert not any("_tc_kernel" in n for n in names), names
    t = qkv.interior().double().reshape(B, N, 3, heads, d).permute(2, 0, 3, 1, 4)
    q, k, v = (t[i].clone().requires_grad_(True) for i in range(3))
    scale = 1.0 / math.sqrt(d)
    o_ref, lse_ref = _attn_ref(q, k, v, scale)
    go = dout.interior().double().reshape(B, N, heads, d).permute(0, 2, 1, 3)
    o_ref.backward(go)
    o = out.interior().double().reshape(B, N, heads, d).permute(0, 2, 1, 3)
    g = dqkv.interior().double().reshape(B, N, 3, heads, d).permute(2, 0, 3, 1, 4)

    def nrel(a, b):
        return float((a - b).norm() / b.norm())
    assert nrel(o, o_ref) < 1.5e-3, nrel(o, o_ref)
    assert float((lse.double() - lse_ref).abs().max()) < 2e-3
    for i, (name, r) in enumerate((("dq", q.grad), ("dk", k.grad), ("dv", v.grad))):
        assert nrel(g[i], r) < 6e-3, (name, nrel(g[i], r))


# ================================================================================================================
# GPU: the dtype rule of the C ABI
# ================================================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("code,want", [(2, 0), (3, DDPM_E_ARG)], ids=["f16", "unknown"])
def test_entry_points_accept_f16_and_reject_unknown_codes(mods, code, want):
    _lib, engine = mods
    L = _lib.lib
    E = engine.Exec(dev(), _lib.F16, True, True)
    N, H, W, Cc = 2, 8, 8, 32
    a, b, o = E.act(N, H, W, Cc), E.act(N, H, W, Cc), E.act(N, H, W, Cc)
    a.interior().normal_()
    b.interior().normal_()
    up = E.act(N, 2 * H, 2 * W, Cc)
    qkv, ao = E.act(N, H, W, 3 * Cc), E.act(N, H, W, Cc)
    sentinel = torch.full((4096,), 7.0, device=dev())
    gamma, beta = torch.ones(Cc, device=dev()), torch.zeros(Cc, device=dev())
    stats = torch.zeros(N, 8, 2, dtype=torch.float64, device=dev())
    lse = torch.zeros(N, 1, H * W, device=dev())
    w = torch.randn(Cc, Cc, 3, 3, device=dev())
    wbuf = torch.zeros(Cc * Cc * 9, dtype=torch.float16, device=dev())
    pred = torch.randn(N, 3 * H * W, device=dev()).half()
    noise = torch.randn_like(pred, dtype=torch.float32)
    tt = torch.tensor([1, 2], device=dev())
    nchw = torch.randn(N, Cc, H, W, device=dev()).half()
    ca = _lib.ConvArgs()
    ca.inp, ca.out = a.desc(), o.desc()
    ca.w, ca.KH, ca.KW, ca.stride, ca.pad, ca.dtype, ca.prefer_tc = wbuf.data_ptr(), 3, 3, 1, 1, code, 1
    wa = _lib.WgradArgs()
    wa.act, wa.dy, wa.dw = a.desc(), b.desc(), sentinel.data_ptr()
    wa.KH = wa.KW = 3
    wa.stride, wa.pad, wa.dtype = 1, 1, code
    snap = [t.buf.t.clone() for t in (o, up, ao)] + [sentinel.clone(), stats.clone(), wbuf.clone()]
    s = _s()
    p = C.c_void_p
    calls = {
        "ddpm_conv": lambda: L.ddpm_conv(C.byref(ca), s),
        "ddpm_gn_stats": lambda: L.ddpm_gn_stats(C.byref(a.desc()), code, 8, p(stats.data_ptr()), s),
        "ddpm_gn_fwd": lambda: L.ddpm_gn_fwd(C.byref(a.desc()), code, 8, p(stats.data_ptr()), p(gamma.data_ptr()), p(beta.data_ptr()),
                                             C.c_float(1e-6), 1, C.c_float(0.0), None, 0, C.byref(o.desc()), s),
        "ddpm_upsample2x": lambda: L.ddpm_upsample2x(C.byref(a.desc()), C.byref(up.desc()), code, s),
        "ddpm_zero_upsample2x": lambda: L.ddpm_zero_upsample2x(C.byref(a.desc()), C.byref(up.desc()), code, s),
        "ddpm_add": lambda: L.ddpm_add(C.byref(a.desc()), C.byref(b.desc()), C.byref(o.desc()), code, s),
        "ddpm_colsum": lambda: L.ddpm_colsum(C.byref(a.desc()), code, None, p(sentinel.data_ptr()), s),
        "ddpm_attn_fwd": lambda: L.ddpm_attn_fwd(C.byref(qkv.desc()), C.byref(ao.desc()), 1, Cc, p(lse.data_ptr()), code, s),
        "ddpm_mse_fwd": lambda: L.ddpm_mse_fwd(p(pred.data_ptr()), code, p(noise.data_ptr()), None, p(sentinel.data_ptr()), N,
                                               3 * H * W, s),
        "ddpm_sinusoid": lambda: L.ddpm_sinusoid(p(tt.data_ptr()), 0, N, 64, p(wbuf.data_ptr()), code, s),
        "ddpm_pack_weights": lambda: L.ddpm_pack_weights(p(w.data_ptr()), Cc, Cc, 3, 3, p(wbuf.data_ptr()), None, code, 0, 0, s),
        "ddpm_nchw_to_nhwc": lambda: L.ddpm_nchw_to_nhwc(p(nchw.data_ptr()), code, Cc, *nchw.stride(), C.byref(o.desc()),
                                                         code, s),
        "ddpm_conv_wgrad": lambda: L.ddpm_conv_wgrad(C.byref(wa), s),
    }
    for name, fn in calls.items():
        if want == 0:
            sentinel.fill_(0.0)
        assert fn() == want, name
    torch.cuda.synchronize()
    if want == DDPM_E_ARG:
        now = [t.buf.t for t in (o, up, ao)] + [sentinel, stats, wbuf]
        for x0, x1 in zip(snap, now):
            assert torch.equal(x0.view(torch.uint8), x1.view(torch.uint8)), "a rejected call wrote"


# ================================================================================================================
# GPU: modules against the fp32 oracle
# ================================================================================================================
LOW_GPU = dict(base_channels=96, channel_mults=(1, 2, 2, 2), num_res_blocks=1, attn_resolutions={8}, num_heads=2,
               head_dim=32, dropout=0.0)


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / b.norm())


@pytest.mark.gpu
def test_unet_autocast_default_dtype_is_fp16_and_beats_bf16():
    """torch.autocast("cuda") with no dtype is fp16: the output is fp16, and its error against the fp32 oracle is at most
    half of the bf16 run's on the same weights and inputs; the same for every parameter gradient of one
    scaler.scale(loss).backward() (divided by the scale).  Parameters whose exact gradient is zero (a convolution bias
    followed by GroupNorm) carry only rounding noise in both runs and are not compared."""
    from oracle import ddpm_oracle as O
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.model.unet_backbone import build_unet_64x64
    torch.manual_seed(0)
    model = build_unet_64x64(**LOW_GPU).to(dev()).train()
    diff = Diffusion(T=1000).to(dev())
    B = 2
    x0 = torch.empty(B, 3, 64, 64, device=dev()).uniform_(-1, 1)
    t = torch.tensor([10, 900], device=dev())
    noise = torch.randn_like(x0)
    spec = O.UNetSpec(in_channels=3, time_embed_dim=512, img_resolution=64, **LOW_GPU)
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    with torch.no_grad():
        y_ref = O.unet_forward(sd, spec, diff.q_sample(x0, t, eps=noise).cpu(), t.cpu())
    _, _, g_ref = O.unet_loss_and_grads(sd, spec, O.make_tables(), x0.cpu(), t.cpu(), noise.cpu())
    res = {}
    for name, kw in (("f16", {}), ("bf16", {"dtype": torch.bfloat16})):
        with torch.no_grad(), torch.autocast("cuda", **kw):
            y = model(diff.q_sample(x0, t, eps=noise), t)
        scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 12)
        for p_ in model.parameters():
            p_.grad = None
        with torch.autocast("cuda", **kw):
            loss = diff.loss_simple(model, x0, t, noise=noise)
        scaler.scale(loss).backward()
        s = float(scaler.get_scale())
        res[name] = (y, {k: p_.grad / s for k, p_ in model.named_parameters()})
    assert res["f16"][0].dtype == torch.float16 and res["bf16"][0].dtype == torch.bfloat16
    e16, eb = _rel(res["f16"][0], y_ref), _rel(res["bf16"][0], y_ref)
    assert e16 <= 0.5 * eb, (e16, eb)
    compared = 0
    for k in g_ref:
        a, b = _rel(res["f16"][1][k], g_ref[k]), _rel(res["bf16"][1][k], g_ref[k])
        if b > 0.3:
            continue
        compared += 1
        assert a <= 0.5 * b, (k, a, b)
    assert compared > len(g_ref) // 2


# ================================================================================================================
# GPU: samplers
# ================================================================================================================
@pytest.mark.gpu
def test_ddim_sampler_fp16_autocast_meets_the_sampler_tolerance():
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.model.unet_backbone import build_unet_64x64
    from ddpm_diffusion_model_b200.testing.ddpim_inference import ddim_infer_sample
    from ddpm_diffusion_model_b200.training_loops.grad_scaler import autocast_ctx
    torch.manual_seed(0)
    model = build_unet_64x64(**LOW_GPU).to(dev()).eval()
    diff = Diffusion(T=1000).to(dev())
    with tempfile.TemporaryDirectory() as d:
        def sample(dt):
            kw = dict(n=8, img_size=64, device="cuda", seed=1234, steps=50, out_path=os.path.join(d, f"{dt}.png"))
            if dt == "fp32":
                return ddim_infer_sample(model, diff, **kw).float()
            with autocast_ctx(dtype=dt):
                return ddim_infer_sample(model, diff, **kw).float()
        ref, g16, gb = sample("fp32"), sample("fp16"), sample("bf16")
    e16, eb = (g16 - ref).abs(), (gb - ref).abs()
    assert float(e16.mean()) <= 2e-3 and float(torch.quantile(e16.flatten()[:2 ** 24], 0.999)) <= 0.1
    assert float(e16.mean()) < float(eb.mean())


@pytest.mark.gpu
def test_ddpm_sampler_fp16_runs_the_folded_upsampling():
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.model.unet_backbone import UNetDenoiser
    from ddpm_diffusion_model_b200.testing.ddpm_inference import ddpm_infer_sample
    cfg = dict(in_channels=3, base_channels=32, channel_mults=(1, 2), num_res_blocks=1, attn_resolutions={8},
               time_embed_dim=64, dropout=0.0, num_heads=2, head_dim=16, img_resolution=16)
    torch.manual_seed(0)
    model = UNetDenoiser(**cfg).to(dev()).eval()
    diff = Diffusion(T=20, img_size=16).to(dev())
    with tempfile.TemporaryDirectory() as d:
        with torch.autocast("cuda", dtype=torch.float16):
            names = [n for n, _ in launched_kernels(lambda: ddpm_infer_sample(model, diff, n=4, img_size=16, device="cuda",
                                                                               out_path=os.path.join(d, "a.png")))]
        ref = ddpm_infer_sample(model, diff, n=4, img_size=16, device="cuda", out_path=os.path.join(d, "b.png"))
        with torch.autocast("cuda", dtype=torch.float16):
            g = ddpm_infer_sample(model, diff, n=4, img_size=16, device="cuda", out_path=os.path.join(d, "c.png"))
    assert any("conv_tc2_f16_kernel<" in n and ", 4, false>" in n for n in names), "folded up-sampling did not run"
    assert torch.isfinite(g).all() and float((g.float() - ref.float()).abs().mean()) < 2e-2


# ================================================================================================================
# GPU: the user AMP loop with torch's GradScaler
# ================================================================================================================
SMALL = dict(in_channels=3, base_channels=32, channel_mults=(1, 2, 2), num_res_blocks=1, attn_resolutions={8},
             time_embed_dim=128, dropout=0.0, num_heads=2, head_dim=16, img_resolution=32)


def _amp_setup():
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.model.unet_backbone import UNetDenoiser
    torch.manual_seed(0)
    model = UNetDenoiser(**SMALL).to(dev()).train()
    diff = Diffusion(T=1000, img_size=32).to(dev())
    gen = torch.Generator().manual_seed(42)
    data = [(torch.empty(8, 3, 32, 32).uniform_(-1, 1, generator=gen).to(dev()), torch.randint(1, 1000, (8,), generator=gen).to(dev()),
             torch.randn(8, 3, 32, 32, generator=gen).to(dev())) for _ in range(3)]
    return model, diff, data


@pytest.mark.gpu
def test_user_amp_loop_follows_the_fp32_trajectory():
    """Three steps of torch.autocast(float16) + GradScaler + AdamW against the same loop in fp32 from the same weights:
    every loss within 1 % (the package's fp32 path matches the fp32 oracle to 1e-4, tests/test_gpu_parity.py)."""
    losses = {}
    for amp in (False, True):
        model, diff, data = _amp_setup()
        opt = torch.optim.AdamW(model.parameters(), lr=1e-3)
        scaler = torch.amp.GradScaler("cuda", enabled=amp)
        out = []
        for x0, t, n in data:
            opt.zero_grad(set_to_none=True)
            with torch.autocast("cuda", dtype=torch.float16, enabled=amp):
                loss = diff.loss_simple(model, x0, t, noise=n)
            scaler.scale(loss).backward()
            scaler.step(opt)
            scaler.update()
            out.append(float(loss))
        losses[amp] = out
    for a, b in zip(losses[True], losses[False]):
        assert abs(a - b) <= 1e-2 * abs(b), (losses[True], losses[False])


@pytest.mark.gpu
def test_grad_scaler_overflow_skips_the_step_and_backs_off():
    model, diff, data = _amp_setup()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3)
    scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 16)
    x0, t, n = data[0]
    with torch.autocast("cuda", dtype=torch.float16):             # one clean step so that the moments exist
        loss = diff.loss_simple(model, x0, t, noise=n)
    scaler.scale(loss).backward()
    scaler.step(opt)
    scaler.update()
    scaler.update(2.0 ** 40)
    params = {k: p.detach().clone() for k, p in model.named_parameters()}
    moments = {k: {s: v.clone() for s, v in opt.state[p].items()} for k, p in model.named_parameters()}
    opt.zero_grad(set_to_none=True)
    x0, t, n = data[1]
    with torch.autocast("cuda", dtype=torch.float16):
        loss = diff.loss_simple(model, x0, t, noise=n)
    scaler.scale(loss).backward()
    assert any(not bool(torch.isfinite(p.grad).all()) for p in model.parameters() if p.grad is not None)
    scaler.step(opt)
    scaler.update()
    assert float(scaler.get_scale()) == 2.0 ** 39
    for k, p in model.named_parameters():
        assert torch.equal(p.detach(), params[k]), k
        assert bool(torch.isfinite(p).all()), k
        for s, v in opt.state[p].items():
            assert torch.equal(v, moments[k][s]), (k, s)
