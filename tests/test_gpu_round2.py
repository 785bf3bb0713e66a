"""Round-2 parity tests: what is TIMED is what is CHECKED.

  * the CelebA256 attention UNet (BASELINE configs[2..4]; reference spec
    `arquitectures/UNetDenoiser arquitecture CelebA256.txt`, full_notebooks/Difussion_Model_CelebHQ.ipynb:1879-1889)
    against the oracle: fp32 forward + loss + every gradient <= 1e-4, bf16 forward <= 2e-2;
  * the low-GPU model's BACKWARD against the oracle (round 1 only checked its forward);
  * the bf16-autocast DDIM sampler that bench.py times, against the fp32 oracle loop with the tolerance of
    BASELINE.md section 4 (mean-abs <= 2e-3, 99.9th percentile <= 0.1 on [0,1] images);
  * render_denoise_strip / render_denoise_strip_ddim (src/testing/ddpm_inference.py:62-119, ddpim_inference.py:108-197);
  * the two advisor findings of round 1 (dropout masks of chained calls, EMA.copy_to after load_state_dict).

The oracle is plain torch; for the 256-px cases it runs on the GPU in fp32 with TF32 switched off (cuDNN's "fp32"
convolutions otherwise carry a 10-bit mantissa and the 1e-4 bar would be meaningless).
"""
import math

import pytest
import torch

from oracle import ddpm_oracle as O

pytestmark = pytest.mark.gpu

LOW_GPU = dict(base_channels=96, channel_mults=(1, 2, 2, 2), num_res_blocks=1, attn_resolutions={8}, num_heads=2, head_dim=32)
CELEBA256 = dict(in_channels=3, base_channels=128, channel_mults=(1, 1, 2, 2, 4), num_res_blocks=2, attn_resolutions={16},
                 time_embed_dim=512, dropout=0.0, num_heads=4, head_dim=64, img_resolution=256)


def dev():
    return torch.device("cuda", 0)


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


@pytest.fixture()
def exact_fp32():
    """fp32 means fp32 for the oracle when it runs on the GPU."""
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _grad_check(model, ref_grads, tol, floor=1e-3):
    gmax = max(float(v.norm()) for v in ref_grads.values())
    worst, worst_k = 0.0, None
    for k, p in model.named_parameters():
        ref = ref_grads[k]
        assert p.grad is not None, k
        e = float((p.grad.detach().double() - ref.double().to(p.grad.device)).norm()) / max(float(ref.norm()), floor * gmax)
        if e > worst:
            worst, worst_k = e, k
    assert worst < tol, (worst_k, worst)
    return worst, worst_k


def test_celeba256_unet_fp32_and_bf16_vs_oracle(exact_fp32):
    """UNetDenoiser(3,128,(1,1,2,2,4),2,{16},512,0.0,4,64,256) at 256 px: 63.1 M parameters, five levels, C=512 -> qkv 768
    -> inner 256 attention, W=256 patches, 24/12-channel GroupNorm groups straddling the concat boundary."""
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.model.unet_backbone import UNetDenoiser
    torch.manual_seed(0)
    kw = dict(CELEBA256)
    model = UNetDenoiser(**kw).to(dev()).train()
    assert sum(p.numel() for p in model.parameters()) == 63100675
    d = Diffusion(T=1000, img_size=256).to(dev())
    B = 1
    x0 = torch.empty(B, 3, 256, 256, device=dev()).uniform_(-1, 1)
    t = torch.tensor([437], device=dev())
    noise = torch.randn_like(x0)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    spec = O.UNetSpec(**kw)
    tb = {k: v.to(dev()) for k, v in O.make_tables().items()}
    ref_loss, ref_eps, ref_g = O.unet_loss_and_grads(sd, spec, tb, x0, t, noise)
    # fp32: forward, loss, every gradient
    loss = d.loss_simple(model, x0, t.clone(), noise=noise)
    loss.backward()
    with torch.no_grad():
        x_t = d.q_sample(x0, t, noise)
        eps = model(x_t, t)
        assert rel(eps, ref_eps) < 1e-4, rel(eps, ref_eps)
        assert abs(float(loss) - float(ref_loss)) < 1e-4 * max(1.0, abs(float(ref_loss)))
        _grad_check(model, ref_g, 1e-4)
        # bf16 autocast (tensor-core path): forward within 2e-2 of the fp32 oracle
        with torch.autocast("cuda", dtype=torch.bfloat16):
            eps_b = model(x_t, t)
        assert eps_b.dtype == torch.bfloat16
        assert rel(eps_b.float(), ref_eps) < 2e-2, rel(eps_b.float(), ref_eps)
    # bf16 backward at 256 px: loss within 2e-2, gradients within the bf16 budget measured on the tiny nets (6e-2 with a
    # 1 % floor, tests/test_gpu_parity.py::test_unet_bf16_attn)
    for p in model.parameters():
        p.grad = None
    with torch.autocast("cuda", dtype=torch.bfloat16):
        loss_b = d.loss_simple(model, x0, t.clone(), noise=noise)
    loss_b.backward()
    assert abs(float(loss_b) - float(ref_loss)) < 2e-2 * max(1.0, abs(float(ref_loss)))
    _grad_check(model, ref_g, 6e-2, floor=1e-2)


def test_low_gpu_model_backward_fp32_vs_oracle(exact_fp32):
    """BASELINE configs[1] model (12.68 M parameters), B=2: loss and every gradient vs the oracle, fp32 <= 1e-4; then the
    bf16-autocast path the benchmark times (tcgen05 fprop/dgrad/wgrad) within the bf16 budget."""
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.model.unet_backbone import build_unet_64x64
    torch.manual_seed(0)
    model = build_unet_64x64(dropout=0.0, **LOW_GPU).to(dev()).train()
    d = Diffusion(T=1000, img_size=64).to(dev())
    x0 = torch.empty(2, 3, 64, 64, device=dev()).uniform_(-1, 1)
    t = torch.tensor([10, 900], device=dev())
    noise = torch.randn_like(x0)
    spec = O.UNetSpec(in_channels=3, time_embed_dim=512, img_resolution=64, dropout=0.0, **LOW_GPU)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    tb = {k: v.to(dev()) for k, v in O.make_tables().items()}
    ref_loss, _, ref_g = O.unet_loss_and_grads(sd, spec, tb, x0, t, noise)
    loss = d.loss_simple(model, x0, t.clone(), noise=noise)
    loss.backward()
    assert abs(float(loss) - float(ref_loss)) < 1e-4 * max(1.0, abs(float(ref_loss)))
    _grad_check(model, ref_g, 1e-4)
    for p in model.parameters():
        p.grad = None
    with torch.autocast("cuda", dtype=torch.bfloat16):
        loss_b = d.loss_simple(model, x0, t.clone(), noise=noise)
    loss_b.backward()
    assert abs(float(loss_b) - float(ref_loss)) < 2e-2 * max(1.0, abs(float(ref_loss)))
    _grad_check(model, ref_g, 6e-2, floor=1e-2)


def _oracle_ddim(model, tb, spec, x, sched, eta=0.0):
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    B = x.shape[0]
    with torch.no_grad():
        for cur, prev in zip(sched[:-1], sched[1:]):
            t = torch.full((B,), int(cur), dtype=torch.long, device=x.device)
            tp = torch.full((B,), int(prev), dtype=torch.long, device=x.device)
            eps = O.unet_forward(sd, spec, x, t)
            x = O.ddim_step(tb, eps, x, t, tp, torch.zeros_like(x), eta, True, None, True)
    return O.to_image01(x)


def test_bf16_autocast_ddim_sampler_vs_fp32_oracle(tmp_path, exact_fp32):
    """`ddim_infer_sample(steps=50, n=8, 64 px)` under bf16 autocast -- the call bench.py times for the DDIM half of the
    metric -- against the fp32 oracle loop from the same x_T.  Tolerance (BASELINE.md section 4, calibrated on the
    reference's own bf16-vs-fp32 deviation: mean 9.5e-4, max 0.21): mean-abs <= 2e-3, 99.9th percentile <= 0.1."""
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.model.unet_backbone import build_unet_64x64
    from ddpm_diffusion_model_b200.testing.ddpim_inference import build_ddim_schedule, ddim_infer_sample
    torch.manual_seed(0)
    model = build_unet_64x64(dropout=0.1, **LOW_GPU).to(dev())
    d = Diffusion(T=1000, img_size=64).to(dev())
    n, steps = 8, 50
    grids = {}
    for name, ctx in (("bf16", torch.autocast("cuda", dtype=torch.bfloat16)), ("fp32", torch.autocast("cuda", enabled=False))):
        with ctx:
            grids[name] = ddim_infer_sample(model, d, n=n, img_size=64, device="cuda", seed=1234, steps=steps, eta=0.0,
                                            out_path=str(tmp_path / f"{name}.png"))
    # the oracle from the same x_T (same seed, same device generator call as testing/_common.initial_noise)
    torch.manual_seed(1234)
    x_T = torch.randn(n, 3, 64, 64, device=dev())
    spec = O.UNetSpec(in_channels=3, time_embed_dim=512, img_resolution=64, dropout=0.0, **LOW_GPU)
    tb = {k: v.to(dev()) for k, v in O.make_tables().items()}
    sched = build_ddim_schedule(d, steps)
    assert sched == O.ddim_schedule_t_linear(1000, steps) and len(sched) - 1 == 49
    img = _oracle_ddim(model.eval(), tb, spec, x_T, sched)
    import torchvision.utils as vutils
    ref_grid = vutils.make_grid(img, nrow=math.ceil(math.sqrt(n)), padding=2)
    e32 = (grids["fp32"] - ref_grid).abs()
    assert float(e32.max()) <= 5e-3, float(e32.max())                        # fp32 sampler tolerance
    e16 = (grids["bf16"].float() - ref_grid).abs().flatten()
    mean_abs, p999 = float(e16.mean()), float(torch.quantile(e16, 0.999))
    assert mean_abs <= 2e-3 and p999 <= 0.1, (mean_abs, p999, float(e16.max()))


def test_denoise_strips_match_step_by_step_trajectories(tmp_path, exact_fp32):
    """render_denoise_strip / render_denoise_strip_ddim: frames are the [0,1] images of the single-sample trajectory at
    the capture steps, assembled with make_grid(nrow=len(frames), padding=pad) -- checked against the oracle's loops fed
    with the same noise draws."""
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.model.unet_backbone import UNetDenoiser
    from ddpm_diffusion_model_b200.testing.ddpim_inference import render_denoise_strip_ddim
    from ddpm_diffusion_model_b200.testing.ddpm_inference import render_denoise_strip
    import torchvision.utils as vutils
    cfg = dict(in_channels=3, base_channels=32, channel_mults=(1, 2), num_res_blocks=1, attn_resolutions={8},
               time_embed_dim=64, dropout=0.0, num_heads=2, head_dim=16, img_resolution=16)
    torch.manual_seed(3)
    model = UNetDenoiser(**cfg).to(dev())
    T = 40
    d = Diffusion(T=T, img_size=16).to(dev())
    spec, tb = O.UNetSpec(**cfg), {k: v.to(dev()) for k, v in O.make_tables(T=T).items()}
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    # ---- DDPM strip
    caps = [39, 30, 20, 10, 5, 0]
    grid = render_denoise_strip(model, d, img_size=16, device="cuda", seed=77, out_path=str(tmp_path / "s.png"), capture_steps=caps, pad=2)
    torch.manual_seed(77)
    x = torch.randn(1, 3, 16, 16, device=dev())
    frames = []
    with torch.no_grad():
        for i in range(T - 1, -1, -1):
            t = torch.full((1,), i, dtype=torch.long, device=dev())
            z = torch.randn_like(x)                                # same draw order as difussion_class.py:186
            x = O.ddpm_step(tb, O.unet_forward(sd, spec, x, t), x, t, z, True, None)
            if i in caps:
                frames.append(O.to_image01(x)[0])
    ref = vutils.make_grid(torch.stack(frames), nrow=len(frames), padding=2)
    assert grid.shape == ref.shape and float((grid.cpu() - ref.cpu()).abs().max()) <= 5e-3
    assert (tmp_path / "s.png").stat().st_size > 0
    # ---- DDIM strip (eta = 0; its own schedule builder: sorted set of round(linspace(T-1, 0, steps)))
    steps = 9
    grid = render_denoise_strip_ddim(model, d, img_size=16, device="cuda", seed=78, out_path=str(tmp_path / "d.png"), steps=steps,
                                     eta=0.0, schedule_kind="linear", pad=1)
    sched = sorted(set(torch.round(torch.linspace(T - 1, 0, steps)).long().tolist()), reverse=True)
    k = min(17, len(sched))
    caps = {sched[i] for i in torch.linspace(0, len(sched) - 1, k).round().long().tolist()}
    torch.manual_seed(78)
    x = torch.randn(1, 3, 16, 16, device=dev())
    frames = []
    with torch.no_grad():
        for i, cur in enumerate(sched):
            prev = sched[i + 1] if i + 1 < len(sched) else 0
            t = torch.full((1,), cur, dtype=torch.long, device=dev())
            tp = torch.full((1,), prev, dtype=torch.long, device=dev())
            x = O.ddim_step(tb, O.unet_forward(sd, spec, x, t), x, t, tp, torch.zeros_like(x), 0.0, True, None, True)
            if cur in caps:
                frames.append(O.to_image01(x)[0])
    ref = vutils.make_grid(torch.stack(frames), nrow=len(frames), padding=1)
    assert grid.shape == ref.shape and float((grid.cpu() - ref.cpu()).abs().max()) <= 5e-3


def test_chained_resblocks_with_dropout_use_their_own_masks_in_backward():
    """Advisor finding (round 1): backward rebuilt the dropout mask from the SHARED {seed, step} counter, so a second
    training-mode forward before backward silently changed the first call's mask.  Chain two ResBlocks (each stand-alone
    call advances the counter) and compare the first block's gradients with a run whose backward directly follows its
    forward (which was always correct)."""
    from ddpm_diffusion_model_b200 import functional as Fn
    from ddpm_diffusion_model_b200.model.unet_backbone import ResBlock
    torch.manual_seed(0)
    b1 = ResBlock(32, 32, 64, dropout=0.3).to(dev()).train()
    b2 = ResBlock(32, 64, 64, dropout=0.3).to(dev()).train()
    x = torch.randn(2, 32, 16, 16, device=dev())
    te = torch.randn(2, 64, device=dev())
    gy = torch.randn(2, 64, 16, 16, device=dev())

    def grads(mod):
        return {k: p.grad.detach().clone() for k, p in mod.named_parameters()}

    # (A) chained: forward b1 (step s+1), forward b2 (step s+2), one backward through both
    Fn.seed_dropout(99, dev())
    xa = x.clone().requires_grad_(True)
    y = b2(b1(xa, te), te)
    y.backward(gy)
    ga, dxa = grads(b1), xa.grad.clone()
    for p in list(b1.parameters()) + list(b2.parameters()):
        p.grad = None
    # (B) same masks (same seed, same step numbers), but every backward directly follows its own forward
    Fn.seed_dropout(99, dev())
    with torch.no_grad():
        y1 = b1(x, te)                                              # step s+1 (mask only matters for y1's value)
    y1d = y1.detach().requires_grad_(True)
    y2 = b2(y1d, te)                                                # step s+2
    assert torch.equal(y2, y)
    y2.backward(gy)
    Fn.seed_dropout(99, dev())
    xb = x.clone().requires_grad_(True)
    y1b = b1(xb, te)                                                # step s+1 again
    assert torch.equal(y1b, y1)
    y1b.backward(y1d.grad)
    gb, dxb = grads(b1), xb.grad
    assert rel(dxa, dxb) < 1e-5, rel(dxa, dxb)
    for k in ga:
        assert rel(ga[k], gb[k]) < 1e-4 or float(gb[k].norm()) < 1e-6, (k, rel(ga[k], gb[k]))
    # a no_grad training-mode forward between forward and backward must not disturb the pending backward either
    Fn.seed_dropout(5, dev())
    xc = x.clone().requires_grad_(True)
    yc = b1(xc, te)
    with torch.no_grad():
        b1(x, te)
    yc.backward(gy[:, :32])
    Fn.seed_dropout(5, dev())
    xd = x.clone().requires_grad_(True)
    b1(xd, te).backward(gy[:, :32])
    assert rel(xc.grad, xd.grad) < 1e-5


def test_ema_copy_to_after_load_state_dict_refreshes_packed_weights(exact_fp32):
    """Advisor finding (round 1): EMA.copy_to's per-tensor branch (used after ema.load_state_dict, before the first
    update) wrote through `.data` without invalidating the packed weight copies -> sampling with `ema=ema` silently used
    the raw weights.  Forward once (packs the weights), swap in a loaded EMA, forward again, compare with the oracle."""
    from ddpm_diffusion_model_b200.model.unet_backbone import UNetDenoiser
    from ddpm_diffusion_model_b200.training_loops.ema import EMA
    cfg = dict(in_channels=3, base_channels=32, channel_mults=(1, 2), num_res_blocks=1, attn_resolutions={8},
               time_embed_dim=64, dropout=0.0, num_heads=2, head_dim=16, img_resolution=16)
    torch.manual_seed(1)
    model = UNetDenoiser(**cfg).to(dev()).eval()
    x = torch.randn(2, 3, 16, 16, device=dev())
    t = torch.tensor([3, 500], device=dev())
    ema = EMA(model, decay=0.99)
    torch.manual_seed(2)
    shadow = [p.detach().clone() + 0.05 * torch.randn_like(p) for p in model.parameters()]
    ema.load_state_dict({"decay": 0.99, "shadow": shadow})
    spec = O.UNetSpec(**cfg)
    for autocast in (False, True):
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
            y_raw = model(x, t)                                     # packs the raw weights
            backup = {k: v.detach().clone() for k, v in model.state_dict().items()}
            ema.copy_to(model)
            y_ema = model(x, t)
            sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
            model.load_state_dict(backup)
            y_back = model(x, t)
        ref = O.unet_forward(sd, spec, x, t)
        tol = 2e-2 if autocast else 1e-4
        assert rel(y_ema.float(), ref) < tol, rel(y_ema.float(), ref)
        assert rel(y_raw.float(), ref) > 5 * tol                    # the swap really changed the function
        assert torch.equal(y_back, y_raw)


def test_grad_norm_diagnostic_uses_the_scale_of_its_own_step():
    """Advisor finding (round 1): FusedStep.grad_norm divided by the scale AFTER ddpm_scaler_update had grown it."""
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.model.unet_backbone import UNetDenoiser
    from ddpm_diffusion_model_b200.training_loops.grad_scaler import make_grad_scaler
    from ddpm_diffusion_model_b200.training_loops import train_one_epoch as T1
    torch.manual_seed(0)
    model = UNetDenoiser(3, 32, (1, 2), 1, {8}, 64, 0.0, 2, 16, 16).to(dev())
    d = Diffusion(T=1000, img_size=16).to(dev())
    opt = torch.optim.AdamW(model.parameters(), lr=1e-4)
    scaler = make_grad_scaler("cuda", True)
    scaler.set_growth_interval(1)                                   # the scale doubles after EVERY clean step
    x = torch.empty(4, 3, 16, 16).uniform_(-1, 1)
    T1.train_one_epoch(model, d, [(x, torch.zeros(4))], opt, scaler=scaler, device="cuda", grad_clip=None)
    fused = model._ddpm_fused_step
    s_after = float(scaler.get_scale())
    st = fused.stats.tolist()
    assert st[2] * 2 == s_after                                     # recorded: the scale before the update
    g = fused.grad_norm(scaler, True)
    assert abs(g - st[0] ** 0.5 / st[2]) < 1e-6 * max(1.0, g) and g > 0


@pytest.mark.parametrize("case", [(2, 32, 32, 8, 8), (3, 192, 192, 16, 16), (2, 192, 192, 32, 32), (1, 128, 128, 128, 128), (5, 64, 64, 4, 4)])
def test_upsample_folded_into_the_conv_gather(case):
    """Upsample = nearest x2 + conv3x3 (unet_backbone.py:56-64) on the tensor-core path: four 2x2-tap phase convolutions
    of the LOW-resolution input with pre-summed weights (DDPM_CONV_UP2X_PHASE) against (i) ATen fp32 on the bf16-rounded
    input and (ii) the materialising path (up-sample kernel + 3x3 convolution), which runs whenever gradients are needed.
    The phase weights are summed in fp32 and rounded once, the reference rounds each of the nine weights: bf16 tolerance
    1e-2."""
    from ddpm_diffusion_model_b200 import _lib, engine
    from ddpm_diffusion_model_b200.model.unet_backbone import Upsample
    import torch.nn.functional as F
    N, Ci, Co, H, W = case
    torch.manual_seed(9)
    mod = Upsample(Ci).to(dev())
    assert mod.conv.out_channels == Co
    E = engine.Exec(dev(), _lib.BF16, False, False)
    x = E.act(N, H, W, Ci); x.interior().normal_()
    wide = E.act(N, 2 * H, 2 * W, Co + 32)                                      # the real target is a slice of the concat buffer
    wide.interior().zero_()                                                     # (pooled buffers come back with old interiors)
    tgt = wide.slice(16, Co)
    n0 = _lib.launch_count(reset=True)
    out, saved = engine.up_fwd(E, mod, x, tgt)
    torch.cuda.synchronize()
    assert _lib.launch_count(reset=True) == 5                                   # the weight pack (first use) + four phase launches
    assert saved is None
    # with gradients the materialising path runs (backward needs the up-sampled tensor anyway; measured: no gain from folding)
    Eg = engine.Exec(dev(), _lib.BF16, True, True)
    out2, u = engine.up_fwd(Eg, mod, x, None)
    torch.cuda.synchronize()
    assert u is not None
    xr = x.interior().float().permute(0, 3, 1, 2)
    ref = F.conv2d(F.interpolate(xr, scale_factor=2, mode="nearest"), mod.conv.weight.detach().bfloat16().float(), mod.conv.bias, padding=1)
    got = out.interior().float().permute(0, 3, 1, 2)
    assert rel(got, ref) < 1e-2, rel(got, ref)
    assert rel(got, out2.interior().float().permute(0, 3, 1, 2)) < 1e-2
    # neighbours of the slice and the halo are untouched
    full = wide.buf.t.float()
    assert float(full[..., :16].abs().max()) == 0 and float(full[..., 16 + Co:].abs().max()) == 0
    assert float(full[:, 0].abs().max() + full[:, -1].abs().max() + full[:, :, 0].abs().max() + full[:, :, -1].abs().max()) == 0


@pytest.mark.parametrize("cin,cout", [(64, 96), (96, 96)])
def test_resblock_backward_inline_and_side_stream_schedules_agree(cin, cout):
    """engine.resblock_bwd with its weight gradients inline on the main stream and on the side stream (Exec.wgrad_side),
    bf16, dropout on, skip convolution and identity skip.  Tensor-core weight gradients are bit-stable; the fp32-atomic
    GroupNorm and bias gradients and the time-bias column sum may reorder."""
    from ddpm_diffusion_model_b200 import _lib, engine
    from ddpm_diffusion_model_b200.model.unet_backbone import ResBlock
    torch.manual_seed(4)
    N, H, W, tdim = 4, 32, 32, 128
    blk = ResBlock(cin, cout, tdim, dropout=0.1).to(dev()).train()
    x = torch.randn(N, cin, H, W, device=dev())
    tb = torch.randn(N, cout, device=dev())
    dy = torch.randn(N, cout, H, W, device=dev())
    rng = torch.tensor([7, 1], dtype=torch.int64, device=dev())
    assert engine.Exec(dev(), _lib.BF16, True, True).wgrad_side                 # the default for bf16
    res = {}
    for side in (False, True):
        for p in blk.parameters():
            p.grad = None
        E = engine.Exec(dev(), _lib.BF16, True, True, rng=rng)
        E.wgrad_side = side
        _, sv = engine.resblock_fwd(E, blk, engine.to_nhwc(E, x), tb, None, 1)
        dx, dtb = engine.resblock_bwd(E, blk, sv, engine.to_nhwc(E, dy))
        torch.cuda.synchronize()
        res[side] = (dx.interior().float(), dtb.clone(),
                     {k: p.grad.clone() for k, p in blk.named_parameters() if p.grad is not None})
    (dx0, dtb0, g0), (dx1, dtb1, g1) = res[False], res[True]
    assert rel(dx1, dx0) <= 1e-6, rel(dx1, dx0)
    assert rel(dtb1, dtb0) <= 1e-6, rel(dtb1, dtb0)
    expect = {"conv1.weight", "conv1.bias", "conv2.weight", "conv2.bias", "norm1.weight", "norm1.bias", "norm2.weight",
              "norm2.bias"} | ({"skip.weight", "skip.bias"} if cin != cout else set())
    assert set(g0) == set(g1) == expect
    for k in expect:
        if k in ("conv1.weight", "conv2.weight", "skip.weight"):
            assert torch.equal(g1[k], g0[k]), k
        else:
            assert rel(g1[k], g0[k]) <= 1e-6, (k, rel(g1[k], g0[k]))


def test_train_one_epoch_stages_pinned_host_batches_ahead_without_changing_results():
    """`train_one_epoch` copies batch i+1 from pinned host memory on a copy stream while step i runs (the reference issues
    `x.to(device, non_blocking=True)` on the compute stream, train_one_epoch.py:63).  Same losses and parameters as with
    device-resident batches, and the loader is not advanced beyond `max_batches`."""
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.model.unet_backbone import UNetDenoiser
    from ddpm_diffusion_model_b200.training_loops.train_one_epoch import last_step_losses, train_one_epoch

    def run(host: bool):
        torch.manual_seed(21)
        model = UNetDenoiser(3, 32, (1, 2), 1, {8}, 64, 0.0, 2, 16, 16).to(dev())
        diff = Diffusion(T=50, img_size=16).to(dev())
        opt = torch.optim.AdamW(model.parameters(), lr=1e-3)
        g = torch.Generator().manual_seed(3)
        batches = [torch.randn(4, 3, 16, 16, generator=g) for _ in range(5)]
        batches = [(b.pin_memory() if host else b.to(dev()), torch.zeros(4)) for b in batches]
        drawn = []

        def loader():
            for k, b in enumerate(batches):
                drawn.append(k)
                yield b
        torch.manual_seed(5)                                  # timesteps / noise of loss_simple
        out = train_one_epoch(model, diff, loader(), opt, scaler=None, ema=None, device="cuda:0", use_autocast=False,
                              max_batches=3)
        return out, last_step_losses().clone(), [p.detach().clone() for p in model.parameters()], drawn

    (a_out, a_loss, a_par, a_drawn), (b_out, b_loss, b_par, b_drawn) = run(True), run(False)
    assert a_out[1:] == b_out[1:] == (3, 12, 3)
    # (the fp32 CUDA-core gradient kernels accumulate with atomics: equal to rounding, not bit for bit)
    assert torch.allclose(a_loss, b_loss, rtol=1e-5, atol=0) and abs(a_out[0] - b_out[0]) < 1e-5
    # parameters: Adam normalises near-zero gradients, so single elements may differ by a step; the tensors agree in norm
    num = sum(float((p - q).double().pow(2).sum()) for p, q in zip(a_par, b_par))
    den = sum(float(q.double().pow(2).sum()) for q in b_par)
    assert (num / den) ** 0.5 < 1e-3
    assert a_drawn == [0, 1, 2] and b_drawn == [0, 1, 2]


def test_train_step_as_cuda_graph_follows_the_eager_trajectory(monkeypatch):
    """The optimiser step captured as ONE CUDA graph (train_one_epoch._GraphStep) against the eager loop on the same seeds:
    the graph draws its timesteps / noise from the same generator sequence, so the per-step losses must track the eager ones
    (bf16 autocast + GradScaler + AdamW + EMA + clip + dropout), the loss trace is complete and ordered, the optimiser's
    step counter advances, and a second epoch replays from its first batch."""
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.model.unet_backbone import UNetDenoiser
    from ddpm_diffusion_model_b200.training_loops.ema import EMA
    from ddpm_diffusion_model_b200.training_loops.grad_scaler import make_grad_scaler
    from ddpm_diffusion_model_b200.training_loops import train_one_epoch as T

    def run(flag: str):
        monkeypatch.setenv("DDPM_B200_TRAIN_GRAPH", flag)
        torch.manual_seed(31)
        model = UNetDenoiser(3, 32, (1, 2), 1, {8}, 64, 0.1, 2, 16, 16).to(dev())
        diff = Diffusion(T=100, img_size=16).to(dev())
        opt = torch.optim.AdamW(model.parameters(), lr=5e-4, weight_decay=0.01)
        ema = EMA(model, decay=0.99)
        scaler = make_grad_scaler("cuda", True)
        g = torch.Generator().manual_seed(9)
        batches = [(torch.randn(8, 3, 16, 16, generator=g).to(dev()), torch.zeros(8)) for _ in range(8)]
        torch.manual_seed(77)
        out1 = T.train_one_epoch(model, diff, batches, opt, scaler=scaler, ema=ema, device="cuda:0", grad_clip=1.0)
        tr1, n1 = T.last_step_losses().clone(), T.last_graph_steps()
        out2 = T.train_one_epoch(model, diff, batches[:5], opt, scaler=scaler, ema=ema, device="cuda:0", grad_clip=1.0, global_step=out1[3])
        tr2, n2 = T.last_step_losses().clone(), T.last_graph_steps()
        step = float(opt.state[next(iter(model.parameters()))]["step"])
        flat = torch.cat([p.detach().float().reshape(-1) for p in model.parameters()])
        shadow = torch.cat([s.detach().float().reshape(-1) for s in ema.shadow])
        return out1, tr1, n1, out2, tr2, n2, step, flat, shadow

    e = run("0")
    e2 = run("0")                                         # eager twice: the run-to-run spread (fp32 atomics in the GroupNorm
    g = run("1")                                          # parameter gradients) that the graph run is allowed
    assert e[2] == 0 and e[5] == 0
    assert g[2] == 0 and g[5] == 5                       # epoch 1 runs eagerly and captures at its end; epoch 2: five replays
    assert g[1].numel() == 8 and g[4].numel() == 5 and e[1].numel() == 8
    assert g[0][1:] == e[0][1:] == (8, 64, 8) and g[3][3] == e[3][3] == 13
    assert e[6] == g[6] == 13.0
    # same RNG sequence => the losses agree step by step (a different timestep / noise draw moves a loss by tens of percent)
    assert torch.allclose(g[1], e[1], rtol=2e-2, atol=2e-3), (g[1], e[1])
    assert torch.allclose(g[4], e[4], rtol=5e-2, atol=5e-3), (g[4], e[4])
    assert abs(g[0][0] - float(g[1].mean())) < 1e-5 and abs(g[3][0] - float(g[4].mean())) < 1e-5
    spread_p = float((e2[7] - e[7]).norm() / e[7].norm())
    spread_s = float((e2[8] - e[8]).norm() / e[8].norm())
    assert float((g[7] - e[7]).norm() / e[7].norm()) < max(3 * spread_p, 1e-3), spread_p
    assert float((g[8] - e[8]).norm() / e[8].norm()) < max(3 * spread_s, 1e-4), spread_s
