"""Attention kernels at long sequences, and a UNet with attention at 32 x 32 / 64 x 64.

  python tools/attn_bench.py kernels          # sweep N x head_dim + the two UNet blocks, tensor-core vs CUDA-core path
  python tools/attn_bench.py blocks           # only the two UNet blocks (for A/B runs against another build)
  python tools/attn_bench.py model --batch 64 # train_one_epoch ms/step and peak allocated memory

Kernel times: CUDA events around many ddpm_attn_fwd / ddpm_attn_bwd calls after warm-up (bf16, halo 1, the NHWC layout
the UNet uses).  Algorithmic TFLOP/s: 4*B*h*N^2*d for the forward, 8*B*h*N^2*d for the backward (the recompute of S
in the backward is overhead, not work).  The CUDA-core path (ddpm_set_force_simt(1)) runs only where its
2*B*h*N^2 fp32 scratch stays under --simt-max-gb.  Set DDPM_B200_LIB to time another build of the library.
"""
import argparse
import ctypes as C
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

SIDES = {64: 8, 256: 16, 576: 24, 1024: 32, 4096: 64, 16384: 128}
TOKENS = 1 << 17                     # B * heads * N of every sweep shape: the same number of query rows everywhere
BLOCKS = [("CelebA256 block", 32, 16, 4, 64), ("low-GPU block", 128, 8, 2, 32)]   # name, B, side, heads, head_dim


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def timed(fn, min_s=0.3, max_iters=200):
    fn(); fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter(); fn(); torch.cuda.synchronize()
    n = max(3, min(max_iters, int(min_s / max(time.perf_counter() - t0, 1e-6))))
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / n          # us per call


def attn_case(_lib, B, side, heads, d, simt):
    dev = torch.device("cuda", 0)
    inner, N = heads * d, side * side

    def buf(c):
        t = torch.zeros(B, side + 2, side + 2, c, dtype=torch.bfloat16, device=dev)
        t[:, 1:-1, 1:-1].normal_()
        return t, _lib.Tensor(t.data_ptr(), B, side, side, c, c, 1)

    (qt, q), (ot, o), (gt, g), (dt_, dq) = buf(3 * inner), buf(inner), buf(inner), buf(3 * inner)
    lse = torch.empty(B, heads, N, device=dev)
    _lib.lib.ddpm_set_force_simt(1 if simt else 0)
    try:
        need = int(_lib.lib.ddpm_attn_bwd_scratch_floats(C.byref(q), C.byref(o), heads, d, _lib.BF16))
        scratch = torch.empty(max(need, 1), device=dev)
        fwd = lambda: _lib.call("ddpm_attn_fwd", C.byref(q), C.byref(o), heads, d, lse.data_ptr(), _lib.BF16, 0)  # noqa: E731
        bwd = lambda: _lib.call("ddpm_attn_bwd", C.byref(q), C.byref(o), C.byref(g), lse.data_ptr(), C.byref(dq),  # noqa: E731
                                heads, d, scratch.data_ptr(), _lib.BF16, 0)
        fwd()
        budget = 0.3 if not simt else 0.05
        return timed(fwd, budget), timed(bwd, budget)
    finally:
        _lib.lib.ddpm_set_force_simt(0)


def row(name, B, side, heads, d, us_f, us_b):
    N = side * side
    ff, fb = 4.0 * B * heads * N * N * d, 8.0 * B * heads * N * N * d
    return f"{name:<22} B={B:<5} N={N:<6} h={heads} d={d:<4} fwd {us_f:10.1f} us {ff / us_f / 1e6:7.1f} TFLOP/s   bwd {us_b:10.1f} us {fb / us_b / 1e6:7.1f} TFLOP/s"


def kernels(args, blocks_only):
    from ddpm_diffusion_model_b200 import _lib
    print(f"# card: {card()}   library: {os.environ.get('DDPM_B200_LIB', _lib.LIB_PATH)}")
    cases = [(n, B, s, h, d) for n, B, s, h, d in BLOCKS]
    if not blocks_only:
        for N, side in SIDES.items():
            for d in (32, 64, 128):
                heads = 4
                cases.append(("sweep", max(1, TOKENS // (N * heads)), side, heads, d))
    for name, B, side, heads, d in cases:
        N = side * side
        f, b = attn_case(_lib, B, side, heads, d, False)
        print("tc     " + row(name, B, side, heads, d, f, b), flush=True)
        if blocks_only:
            continue
        gb = 2 * B * heads * N * N * 4 / 1e9
        if gb > args.simt_max_gb:
            print(f"simt   {name:<22} B={B:<5} N={N:<6} h={heads} d={d:<4} not run: scratch {gb:.1f} GB", flush=True)
        else:
            f, b = attn_case(_lib, B, side, heads, d, True)
            print("simt   " + row(name, B, side, heads, d, f, b), flush=True)
        torch.cuda.empty_cache()


def model(args):
    from ddpm_diffusion_model_b200 import _lib
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.model.unet_backbone import UNetDenoiser
    from ddpm_diffusion_model_b200.training_loops.ema import EMA
    from ddpm_diffusion_model_b200.training_loops.grad_scaler import make_grad_scaler
    from ddpm_diffusion_model_b200.training_loops.train_one_epoch import train_one_epoch
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    m = UNetDenoiser(img_resolution=64, attn_resolutions={32, 16, 8}).to(dev)
    opt = torch.optim.AdamW(m.parameters(), lr=2e-4)
    diff = Diffusion(T=1000, img_size=64).to(dev)
    kw = dict(scaler=make_grad_scaler("cuda", True), ema=EMA(m, decay=0.9995), device="cuda:0", grad_clip=1.0)
    x = torch.empty(args.batch, 3, 64, 64, device=dev).uniform_(-1, 1)
    y = torch.zeros(args.batch)
    train_one_epoch(m, diff, [(x, y)] * 3, opt, **kw)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    train_one_epoch(m, diff, [(x, y)] * args.steps, opt, **kw)
    b.record()
    torch.cuda.synchronize()
    print(f"# card: {card()}   library: {os.environ.get('DDPM_B200_LIB', _lib.LIB_PATH)}")
    print(f"model  UNetDenoiser(img_resolution=64, attn_resolutions={{32,16,8}}) B={args.batch}: "
          f"{a.elapsed_time(b) / args.steps:8.2f} ms/step over {args.steps} steps, "
          f"peak allocated {torch.cuda.max_memory_allocated() / 2**30:6.2f} GiB", flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("mode", choices=["kernels", "blocks", "model"])
    ap.add_argument("--simt-max-gb", type=float, default=24.0)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--steps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("attn_bench: needs a CUDA device")
    if args.mode == "model":
        model(args)
    else:
        kernels(args, args.mode == "blocks")


if __name__ == "__main__":
    main()
