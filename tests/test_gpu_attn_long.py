"""Attention on the tensor cores beyond 256 tokens: the key-tiled online-softmax forward and the tiled backward of
csrc/attn_tc.cu (head_dim 32 / 64 / 128, any H x W with W <= 128, ragged and partial tiles).

Kernel outputs are compared with a float64 reference computed on the GPU from the same bf16-rounded inputs: relative
Frobenius error <= 2e-2 (the bf16 bar of tests/test_gpu_parity.py::test_attention_fwd_bwd), lse within 1e-3.
Every test needs a GPU except the last, which checks the scratch-size arithmetic on the host.
"""
import ctypes as C

import pytest
import torch

gpu = pytest.mark.gpu

SHAPES = [  # B, H, W, heads, head_dim
    (2, 32, 32, 4, 64), (1, 64, 64, 2, 64), (1, 128, 128, 1, 64),
    (2, 24, 24, 2, 32), (1, 20, 20, 3, 128), (3, 9, 9, 2, 64),        # ragged tiles (R*W < 128, N % 16 != 0)
    (1, 48, 40, 2, 32),                                                # non-square
    (2, 16, 16, 4, 128),                                               # single tile, head_dim 128
]
CUDA_CORE_KERNELS = ("attn_fwd_kernel", "attn_bwd_q_kernel", "attn_bwd_kv_kernel")
TC_KERNELS = ("attn_fwd_tc_kernel", "attn_bwd_dq_tc_kernel", "attn_bwd_dkv_tc_kernel")


def dev():
    return torch.device("cuda", 0)


def rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / (b.norm() + 1e-30))


@pytest.fixture(scope="module")
def lib():
    from ddpm_diffusion_model_b200 import _lib
    _lib.lib.ddpm_set_force_simt(0)
    return _lib


class Buf:
    """A bf16 NHWC buffer with a halo ring and `pad` channels of pitch padding, both filled with `fill`."""

    def __init__(self, lib, x, halo, pad, fill):
        B, H, W, Cc = x.shape
        self.t = torch.full((B, H + 2 * halo, W + 2 * halo, Cc + pad), fill, dtype=torch.bfloat16, device=dev())
        self.halo, self.C = halo, Cc
        self.inner().copy_(x)
        self.desc = lib.Tensor(self.t.data_ptr(), B, H, W, Cc, Cc + pad, halo)

    def inner(self):
        h = self.halo
        return self.t[:, h:self.t.shape[1] - h, h:self.t.shape[2] - h, :self.C]


def inputs(B, H, W, heads, d, seed):
    g = torch.Generator(device=dev()).manual_seed(seed)
    qkv = torch.randn(B, H, W, 3 * heads * d, device=dev(), generator=g)
    dout = torch.randn(B, H, W, heads * d, device=dev(), generator=g)
    return qkv.bfloat16(), dout.bfloat16()


def run(lib, qkv, dout, heads, d, halo=1, pad=0, fill=0.0):
    B, H, W, _ = qkv.shape
    N = H * W
    q, o = Buf(lib, qkv, halo, pad, fill), Buf(lib, torch.zeros(B, H, W, heads * d, device=dev()), halo, pad, fill)
    go, dq = Buf(lib, dout, halo, pad, fill), Buf(lib, torch.zeros(B, H, W, 3 * heads * d, device=dev()), halo, pad, fill)
    lse = torch.empty(B, heads, N, device=dev())
    lib.call("ddpm_attn_fwd", C.byref(q.desc), C.byref(o.desc), heads, d, lse.data_ptr(), lib.BF16, 0)
    need = int(lib.lib.ddpm_attn_bwd_scratch_floats(C.byref(q.desc), C.byref(o.desc), heads, d, lib.BF16))
    scratch = torch.empty(max(need, 1), device=dev())
    lib.call("ddpm_attn_bwd", C.byref(q.desc), C.byref(o.desc), C.byref(go.desc), lse.data_ptr(), C.byref(dq.desc),
             heads, d, scratch.data_ptr(), lib.BF16, 0)
    torch.cuda.synchronize()
    return dict(o=o, lse=lse, dqkv=dq, need=need)


def reference(qkv, dout, heads, d):
    """float64 attention forward / backward of the bf16 inputs, in the kernels' NHWC channel layout."""
    B, H, W, _ = qkv.shape
    N = H * W
    x = qkv.double().reshape(B, N, 3, heads, d).permute(2, 0, 3, 1, 4)          # [3][B][heads][N][d]
    q, k, v = x[0], x[1], x[2]
    g = dout.double().reshape(B, N, heads, d).transpose(1, 2)
    scale = d ** -0.5
    s = (q @ k.transpose(-1, -2)) * scale
    lse = torch.logsumexp(s, -1)
    p = torch.exp(s - lse[..., None])
    del s
    o = p @ v
    dv = p.transpose(-1, -2) @ g
    ds = p * (g @ v.transpose(-1, -2) - (g * o).sum(-1, keepdim=True))
    del p
    dq, dk = (ds @ k) * scale, (ds.transpose(-1, -2) @ q) * scale
    nhwc = lambda t: t.transpose(1, 2).reshape(B, H, W, heads * d)  # noqa: E731
    return dict(o=nhwc(o), lse=lse, dqkv=torch.cat([nhwc(dq), nhwc(dk), nhwc(dv)], -1))


def check(got, ref, heads, d, grads=("dq", "dk", "dv")):
    inner = heads * d
    o, dqkv = got["o"].inner().float(), got["dqkv"].inner().float()
    assert torch.isfinite(o).all() and torch.isfinite(dqkv).all() and torch.isfinite(got["lse"]).all()
    assert rel(o, ref["o"]) < 2e-2, rel(o, ref["o"])
    lse_err = float((got["lse"].double() - ref["lse"]).abs().max())
    assert lse_err < 1e-3, lse_err
    for i, name in enumerate(("dq", "dk", "dv")):
        if name not in grads:
            continue
        e = rel(dqkv[..., i * inner:(i + 1) * inner], ref["dqkv"][..., i * inner:(i + 1) * inner])
        assert e < 2e-2, (name, e)


@gpu
@pytest.mark.parametrize("halo", [1, 0], ids=["halo1", "halo0"])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_kernels_vs_fp64(lib, shape, halo):
    B, H, W, heads, d = shape
    qkv, dout = inputs(B, H, W, heads, d, seed=H * W + d)
    got = run(lib, qkv, dout, heads, d, halo=halo)
    check(got, reference(qkv, dout, heads, d), heads, d)


@gpu
@pytest.mark.parametrize("shape", [(1, 32, 32, 2, 64), (2, 20, 20, 1, 128), (1, 24, 24, 2, 32)], ids=lambda s: "x".join(map(str, s)))
def test_online_softmax_stress(lib, shape):
    """Logits spanning > 80 with every row's maximum in the last key tile: each new tile raises the running max, so a
    missing or wrong rescale of o and l either overflows or loses the row.  dq is not compared: with the probability mass
    on keys that differ only slightly, dq = scale * sum_j dS_j k_j cancels to ~2 % of its terms, and the bf16 rounding of
    dS (2^-9) is amplified beyond the 2e-2 bar in any bf16 backward; the backward has no online rescale to stress."""
    B, H, W, heads, d = shape
    N, inner = H * W, heads * d
    g = torch.Generator(device=dev()).manual_seed(7)
    qkv = torch.randn(B, H, W, 3 * inner, device=dev(), generator=g)
    # keys grow along the token order: k_j = ramp(j) * u + noise, q = 12 * u  ->  logit(i, j) rises with j
    u = torch.randn(heads, d, device=dev(), generator=g)
    u = u / u.norm(dim=-1, keepdim=True)
    ramp = torch.linspace(-1.0, 1.0, N, device=dev()).reshape(1, H, W, 1, 1)
    k = ramp * u * (d ** 0.5) * 4.0 + 0.1 * qkv[..., inner:2 * inner].reshape(B, H, W, heads, d)
    qkv[..., :inner] = (12.0 * u).expand(B, H, W, heads, d).reshape(B, H, W, inner)
    qkv[..., inner:2 * inner] = k.reshape(B, H, W, inner)
    qkv, dout = qkv.bfloat16(), torch.randn(B, H, W, inner, device=dev(), generator=g).bfloat16()
    ref = reference(qkv, dout, heads, d)
    x = qkv.double().reshape(B, N, 3, heads, d)
    logits = torch.einsum("bnhd,bmhd->bhnm", x[:, :, 0], x[:, :, 1]) * d ** -0.5
    span = logits.amax(-1) - logits.amin(-1)
    assert float(span.min()) > 80, float(span.min())
    last_tile = (H - 1) // (128 // W) * (128 // W) * W                     # first token of the last key tile
    assert bool((logits.argmax(-1) >= last_tile).all())
    got = run(lib, qkv, dout, heads, d)
    check(got, ref, heads, d, grads=("dk", "dv"))
    assert torch.isfinite(got["dqkv"].inner().float()).all()


@gpu
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_nan_fences(lib, shape):
    """Halo pixels and pitch padding of every buffer hold NaN: no TMA box, mask or store may touch them."""
    B, H, W, heads, d = shape
    qkv, dout = inputs(B, H, W, heads, d, seed=H * W + d)
    got = run(lib, qkv, dout, heads, d, halo=1, pad=8, fill=float("nan"))
    check(got, reference(qkv, dout, heads, d), heads, d)
    for buf in (got["o"], got["dqkv"]):            # and the kernels wrote nothing outside the logical tensor
        t = buf.t.float()
        inside = torch.zeros_like(t, dtype=torch.bool)
        inside[:, 1:-1, 1:-1, :buf.C] = True
        assert bool(torch.isnan(t[~inside]).all())


@gpu
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_tensor_core_path_ran(lib, shape):
    from torch.profiler import ProfilerActivity, profile
    B, H, W, heads, d = shape
    qkv, dout = inputs(B, H, W, heads, d, seed=1)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        got = run(lib, qkv, dout, heads, d)
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    for k in TC_KERNELS:
        assert any(k in n for n in names), (k, sorted(set(names)))
    assert not [n for n in names if any(k in n for k in CUDA_CORE_KERNELS)]
    assert got["need"] == B * heads * H * W


@gpu
def test_attn_block_memory_at_64x64():
    """An AttnBlock training step at 64 x 64 (N = 4096): no N x N buffer.  The CUDA-core backward needed
    2 * B * heads * N^2 fp32 of scratch; peak memory now grows by less than a quarter of that."""
    from ddpm_diffusion_model_b200.model.attention import AttnBlock
    B, heads, N = 8, 4, 64 * 64
    torch.manual_seed(0)
    blk = AttnBlock(256, heads, 64).to(dev()).train()
    x = torch.randn(B, 256, 64, 64, device=dev(), requires_grad=True)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        blk(x).float().sum().backward()             # warm-up: weight caches, pools
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    with torch.autocast("cuda", dtype=torch.bfloat16):
        y = blk(x)
    y.float().sum().backward()
    torch.cuda.synchronize()
    grown = torch.cuda.max_memory_allocated() - base
    assert grown < 0.25 * 2 * B * heads * N * N * 4, grown
    assert torch.isfinite(x.grad).all()


MODELS = [  # attention at 64^2 and 32^2 (head_dim 32); at 32^2 with head_dim 128
    dict(in_channels=3, base_channels=32, channel_mults=(1, 2), num_res_blocks=1, attn_resolutions={64, 32},
         time_embed_dim=64, dropout=0.0, num_heads=2, head_dim=32, img_resolution=64),
    dict(in_channels=3, base_channels=32, channel_mults=(1, 2), num_res_blocks=1, attn_resolutions={32},
         time_embed_dim=64, dropout=0.0, num_heads=1, head_dim=128, img_resolution=32),
]


@gpu
@pytest.mark.parametrize("cfg", MODELS, ids=["attn64_32_d32", "attn32_d128"])
def test_unet_long_attention_vs_oracle(cfg):
    """bf16-autocast forward and every parameter gradient against the fp32 oracle, with the bars of the bf16 UNet case
    (tests/test_gpu_parity.py::test_unet_bf16_attn): 2e-2 forward, 6e-2 gradients with a 1 % floor."""
    from oracle import ddpm_oracle as O
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.model.unet_backbone import UNetDenoiser
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        torch.manual_seed(0)
        S = cfg["img_resolution"]
        model = UNetDenoiser(**cfg).to(dev()).train()
        d = Diffusion(T=1000, img_size=S).to(dev())
        x0 = torch.empty(2, 3, S, S, device=dev()).uniform_(-1, 1)
        t = torch.tensor([37, 801], device=dev())
        noise = torch.randn_like(x0)
        sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
        tb = {k: v.to(dev()) for k, v in O.make_tables().items()}
        ref_loss, ref_eps, ref_g = O.unet_loss_and_grads(sd, O.UNetSpec(**cfg), tb, x0, t, noise)
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            eps = model(d.q_sample(x0, t, noise), t)
        assert rel(eps.float(), ref_eps) < 2e-2, rel(eps.float(), ref_eps)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            loss = d.loss_simple(model, x0, t.clone(), noise=noise)
        loss.backward()
        assert abs(float(loss) - float(ref_loss)) < 2e-2 * max(1.0, abs(float(ref_loss)))
        gmax = max(float(v.norm()) for v in ref_g.values())
        worst, worst_k = 0.0, None
        for k, p in model.named_parameters():
            ref = ref_g[k].double().to(dev())
            e = float((p.grad.double() - ref).norm()) / max(float(ref.norm()), 1e-2 * gmax)
            if e > worst:
                worst, worst_k = e, k
        assert worst < 6e-2, (worst_k, worst)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


@gpu
def test_bwd_rejects_ineligible_dout(lib):
    """qkv / out on the tensor-core path but dout with another halo: the scratch was sized for the tensor-core kernels
    (B * heads * N floats), so the call must fail instead of running the CUDA-core kernels' N x N writes into it."""
    B, H, W, heads, d = 1, 32, 32, 2, 64
    qkv, dout = inputs(B, H, W, heads, d, seed=3)
    q, o = Buf(lib, qkv, 1, 0, 0.0), Buf(lib, torch.zeros(B, H, W, heads * d, device=dev()), 1, 0, 0.0)
    go = Buf(lib, dout, 0, 0, 0.0)
    dq = Buf(lib, torch.zeros(B, H, W, 3 * heads * d, device=dev()), 1, 0, 0.0)
    lse = torch.empty(B, heads, H * W, device=dev())
    lib.call("ddpm_attn_fwd", C.byref(q.desc), C.byref(o.desc), heads, d, lse.data_ptr(), lib.BF16, 0)
    need = int(lib.lib.ddpm_attn_bwd_scratch_floats(C.byref(q.desc), C.byref(o.desc), heads, d, lib.BF16))
    assert need == B * heads * H * W
    scratch = torch.full((need + 1024,), 7.0, device=dev())
    before = dq.t.clone()
    torch.cuda.synchronize()
    with pytest.raises(RuntimeError, match="rejected its arguments"):
        lib.call("ddpm_attn_bwd", C.byref(q.desc), C.byref(o.desc), C.byref(go.desc), lse.data_ptr(), C.byref(dq.desc),
                 heads, d, scratch.data_ptr(), lib.BF16, 0)
    torch.cuda.synchronize()
    assert torch.equal(dq.t, before)
    assert bool((scratch == 7.0).all())


@pytest.mark.parametrize("case", [
    # (B, H, W, heads, d, dtype, tensor-core)
    (2, 64, 64, 4, 128, "bf16", True), (1, 128, 128, 1, 64, "bf16", True), (3, 9, 9, 2, 32, "bf16", True),
    (2, 64, 64, 4, 64, "f32", False), (2, 32, 32, 2, 16, "bf16", False), (1, 4, 256, 1, 64, "bf16", False),
])
def test_bwd_scratch_floats_host_only(case):
    """ddpm_attn_bwd_scratch_floats is host arithmetic on descriptors (no device memory is touched): B*heads*N floats for
    the tensor-core backward, 2*B*heads*N^2 for the CUDA-core one (fp32, head_dim 16, W = 256)."""
    from ddpm_diffusion_model_b200 import _lib
    B, H, W, heads, d, dt, tc = case
    dtype = _lib.BF16 if dt == "bf16" else _lib.F32
    qkv = _lib.Tensor(1 << 20, B, H, W, 3 * heads * d, 3 * heads * d, 1)
    out = _lib.Tensor(1 << 21, B, H, W, heads * d, heads * d, 1)
    _lib.lib.ddpm_set_force_simt(0)
    got = int(_lib.lib.ddpm_attn_bwd_scratch_floats(C.byref(qkv), C.byref(out), heads, d, dtype))
    N = H * W
    assert got == (B * heads * N if tc else 2 * B * heads * N * N)


