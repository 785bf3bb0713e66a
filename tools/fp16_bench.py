"""fp16 against bf16, alternating in one process: the tensor-core kernels, GroupNorm, a UNet train step and DDIM sampling.

  python tools/fp16_bench.py [--reps 5]

Each measurement runs the fp16 and the bf16 build of the same work back to back, `--reps` times, and reports the median of
each and their ratio.  Kernel times are CUDA events around many launches after warm-up (inputs are rewritten by nothing
in between: the conv working sets of B = 128 exceed the 126 MB L2, the GroupNorm ones at 96@64 do too).  Shapes:
  * conv fprop / dgrad / wgrad: bench.py's conv_roofline rows (3x3 s1 of the low-GPU UNet), B = 128;
  * GroupNorm + SiLU forward / backward (dropout 0.1) at 96 channels @ 64 px and 256 channels @ 256 px;
  * the CelebA256 attention block (B 32, 16 x 16 tokens, 4 heads of 64) forward and backward;
  * a UNet (low-GPU config, 64 px, B = 128) forward + backward with the user AMP loop (autocast + GradScaler + AdamW);
  * ddim_infer_sample(steps=100) at B = 256, 64 px.
The card name and power limit are printed first: every number here belongs to that card at that limit.
"""
import argparse
import ctypes as C
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

CONV_SHAPES = [(96, 96, 64, 5), (192, 192, 32, 5), (192, 192, 64, 1), (288, 96, 64, 1), (384, 192, 32, 1),
               (192, 192, 16, 6), (192, 192, 8, 9), (96, 192, 32, 1), (384, 192, 16, 1)]
LOW_GPU = dict(base_channels=96, channel_mults=(1, 2, 2, 2), num_res_blocks=1, attn_resolutions={8}, num_heads=2,
               head_dim=32, dropout=0.1)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def event_time(fn, iters):
    fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / iters * 1e3          # us


def ab(name, make, reps, iters):
    """make(dt_code) -> callable; alternates fp16 / bf16 `reps` times.  Prints and returns (fp16 us, bf16 us)."""
    from ddpm_diffusion_model_b200 import _lib
    fns = {d: make(d) for d in (_lib.F16, _lib.BF16)}
    t = {d: [] for d in fns}
    for _ in range(reps):
        for d in (_lib.F16, _lib.BF16):
            t[d].append(event_time(fns[d], iters))
    a, b = statistics.median(t[_lib.F16]), statistics.median(t[_lib.BF16])
    print(f"{name:44s} fp16 {a:10.1f} us   bf16 {b:10.1f} us   fp16/bf16 {a / b:6.3f}", flush=True)
    return a, b


def conv_fn(dt, ci, co, hw, B, op):
    from ddpm_diffusion_model_b200 import engine
    E = engine.Exec(torch.device("cuda"), dt, True, True)
    w = torch.nn.Parameter(torch.randn(co, ci, 3, 3, device="cuda") * 0.02)
    x = E.act(B, hw, hw, ci)
    x.interior().normal_()
    y = E.act(B, hw, hw, co)
    y.interior().normal_()
    if op == "fprop":
        wf, _ = E.wcache.get(E, w, dt, False)
        return lambda: engine.conv(E, x, wf, y, 3, 1, 1)
    if op == "dgrad":
        _, wd = E.wcache.get(E, w, dt, True)
        return lambda: engine.conv(E, y, wd, x, 3, 1, 1)
    w.grad = torch.zeros_like(w)
    b = torch.nn.Parameter(torch.zeros(co, device="cuda"))
    b.grad = torch.zeros_like(b)
    return lambda: engine.wgrad(E, x, y, w, 3, 1, 1, bias=b)


def gn_fn(dt, Cc, hw, B, bwd):
    from ddpm_diffusion_model_b200 import _lib, engine
    E = engine.Exec(torch.device("cuda"), dt, True, True)
    L = _lib.lib
    x, o, dy = E.act(B, hw, hw, Cc), E.act(B, hw, hw, Cc), E.act(B, hw, hw, Cc)
    x.interior().normal_()
    dy.interior().normal_()
    g, bt = torch.ones(Cc, device="cuda"), torch.zeros(Cc, device="cuda")
    dg, db = torch.zeros(Cc, device="cuda"), torch.zeros(Cc, device="cuda")
    st = torch.zeros(B, 32, 2, dtype=torch.float64, device="cuda")
    rng = torch.tensor([1, 1], dtype=torch.int64, device="cuda")
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = C.c_void_p
    fwd = lambda: L.ddpm_gn_fwd(C.byref(x.desc()), dt, 32, p(st.data_ptr()), p(g.data_ptr()), p(bt.data_ptr()),  # noqa: E731
                                C.c_float(1e-6), 1, C.c_float(0.1), p(rng.data_ptr()), 1, C.byref(o.desc()), s)
    if not bwd:
        return fwd
    fwd()
    return lambda: L.ddpm_gn_bwd_colsum(C.byref(x.desc()), dt, 32, p(st.data_ptr()), p(g.data_ptr()), p(bt.data_ptr()),
                                        C.c_float(1e-6), 1, C.c_float(0.1), p(rng.data_ptr()), 1, C.byref(dy.desc()),
                                        C.byref(o.desc()), 0, p(dg.data_ptr()), p(db.data_ptr()), None, None, 0, s)


def attn_fn(dt, bwd, B=32, side=16, heads=4, d=64):
    from ddpm_diffusion_model_b200 import _lib, engine
    E = engine.Exec(torch.device("cuda"), dt, True, True)
    L = _lib.lib
    inner = heads * d
    qkv, out, dout, dqkv = E.act(B, side, side, 3 * inner), E.act(B, side, side, inner), E.act(B, side, side, inner), \
        E.act(B, side, side, 3 * inner)
    qkv.interior().normal_()
    dout.interior().normal_()
    lse = torch.empty(B, heads, side * side, device="cuda")
    scr = torch.empty(int(L.ddpm_attn_bwd_scratch_floats(C.byref(qkv.desc()), C.byref(out.desc()), heads, d, dt)), device="cuda")
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    fwd = lambda: L.ddpm_attn_fwd(C.byref(qkv.desc()), C.byref(out.desc()), heads, d, C.c_void_p(lse.data_ptr()), dt, s)  # noqa: E731
    if not bwd:
        return fwd
    fwd()
    return lambda: L.ddpm_attn_bwd(C.byref(qkv.desc()), C.byref(out.desc()), C.byref(dout.desc()), C.c_void_p(lse.data_ptr()),
                                   C.byref(dqkv.desc()), heads, d, C.c_void_p(scr.data_ptr()), dt, s)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--batch", type=int, default=128)
    args = ap.parse_args()
    from ddpm_diffusion_model_b200 import _lib
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.model.unet_backbone import build_unet_64x64
    from ddpm_diffusion_model_b200.testing.ddpim_inference import ddim_infer_sample
    print("card (name, power limit, max SM clock):", card(), flush=True)
    B, R = args.batch, args.reps
    tot = {"fprop": [0.0, 0.0], "dgrad": [0.0, 0.0], "wgrad": [0.0, 0.0]}
    for op in ("fprop", "dgrad", "wgrad"):
        for ci, co, hw, cnt in CONV_SHAPES:
            a, b = ab(f"conv {op} {ci}->{co}@{hw} B={B}", lambda dt: conv_fn(dt, ci, co, hw, B, op), R, 10)
            tot[op][0] += cnt * a
            tot[op][1] += cnt * b
        print(f"{'conv ' + op + ' count-weighted total':44s} fp16 {tot[op][0]:10.1f} us   bf16 {tot[op][1]:10.1f} us   "
              f"fp16/bf16 {tot[op][0] / tot[op][1]:6.3f}", flush=True)
    for Cc, hw, nb in ((96, 64, B), (256, 256, 16)):
        for bwd in (False, True):
            ab(f"groupnorm+silu+dropout {'bwd' if bwd else 'fwd'} {Cc}@{hw} B={nb}", lambda dt: gn_fn(dt, Cc, hw, nb, bwd), R, 20)
    for bwd in (False, True):
        ab(f"attention CelebA256 block {'bwd' if bwd else 'fwd'}", lambda dt: attn_fn(dt, bwd), R, 50)

    torch.manual_seed(0)
    model = build_unet_64x64(**LOW_GPU).cuda().train()
    diff = Diffusion(T=1000).cuda()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-4, fused=True)
    scaler = torch.amp.GradScaler("cuda")
    x0 = torch.empty(B, 3, 64, 64, device="cuda").uniform_(-1, 1)
    t = torch.randint(1, 1000, (B,), device="cuda")
    n = torch.randn_like(x0)
    tdt = {_lib.F16: torch.float16, _lib.BF16: torch.bfloat16}

    def step(dt):
        def run():
            opt.zero_grad(set_to_none=True)
            with torch.autocast("cuda", dtype=tdt[dt]):
                loss = diff.loss_simple(model, x0, t, noise=n)
            scaler.scale(loss).backward()
            scaler.step(opt)
            scaler.update()
        return run
    ab(f"UNet low-GPU 64px B={B} AMP train step", step, R, 5)
    model.eval()
    with tempfile.TemporaryDirectory() as d:
        def sample(dt):
            def run():
                with torch.autocast("cuda", dtype=tdt[dt]):
                    ddim_infer_sample(model, diff, n=256, img_size=64, device="cuda", steps=100, seed=1,
                                      out_path=os.path.join(d, "s.png"))
            return run
        ab("ddim_infer_sample steps=100 B=256 64px", sample, max(2, R // 2), 1)


if __name__ == "__main__":
    main()
