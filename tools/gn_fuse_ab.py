"""GroupNorm-in-the-operand-path A/B (run under gpurun).

Per layer shape: [ddpm_gn_fwd + ddpm_conv] against [ddpm_gn_coeffs + ddpm_conv(gn_ab)] and each launch alone, CUDA events;
then DDIM-100 through ddim_infer_sample with DDPM_B200_FUSE_GN=0 / 1 in one process.

    python tools/gn_fuse_ab.py [--batch 256] [--no-ddim] [--c256]
"""
import argparse, contextlib, io, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from ddpm_diffusion_model_b200 import _lib, engine

ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=256)
ap.add_argument("--reps", type=int, default=10)
ap.add_argument("--no-ddim", action="store_true")
ap.add_argument("--no-layers", action="store_true")
ap.add_argument("--c256", action="store_true")
ap.add_argument("--shape", default=None, help="one 'Cin,Cout,H,k' (for ncu)")
args = ap.parse_args()
dev = torch.device("cuda", 0)
B = args.batch


def timeit(fn, reps=None):
    reps = reps or args.reps
    fn(); fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / reps * 1e3        # us


SHAPES = [(96, 96, 64, 3), (192, 192, 32, 3), (288, 96, 64, 3), (192, 192, 64, 3), (384, 192, 32, 3), (192, 192, 16, 3),
          (192, 192, 8, 3), (384, 192, 16, 3), (192, 576, 16, 1)]
if args.shape:
    SHAPES = [tuple(int(v) for v in args.shape.split(","))]
if not args.no_layers:
    E = engine.Exec(dev, _lib.BF16, False, False)
    print(f"B={B}: us per launch; pair = GroupNorm(+SiLU) + conv", flush=True)
    print(f"{'shape':>18s} {'gn_fwd':>8s} {'conv':>8s} {'sum':>8s} | {'coeffs':>8s} {'conv_gn':>8s} {'sum':>8s} | saved", flush=True)
    for (Ci, Co, H, k) in SHAPES:
        torch.manual_seed(0)
        gn = torch.nn.GroupNorm(32, Ci).to(dev)
        w = torch.nn.Parameter(torch.randn(Co, Ci, k, k, device=dev) / (Ci * k * k) ** 0.5)
        b = torch.randn(Co, device=dev)
        wf, _ = E.wcache.get(E, w, _lib.BF16, False)
        x = E.act(B, H, H, Ci); x.interior().normal_()
        a = E.act(B, H, H, Ci); y = E.act(B, H, H, Co)
        act = 1 if k == 3 else 0
        t_gn = timeit(lambda: engine.gn_fwd(E, x, gn, act, 0.0, 0, out=a))
        t_cv = timeit(lambda: engine.conv(E, a, wf, y, k, 1, k // 2, bias=b))
        ab = engine.gn_coeffs(E, x, gn)
        t_co = timeit(lambda: engine.gn_coeffs(E, x, gn))
        t_cg = timeit(lambda: engine.conv(E, x, wf, y, k, 1, k // 2, bias=b, gn_ab=ab, gn_act=act))
        print(f"{Ci:4d}->{Co:3d}@{H:<3d}k{k}   {t_gn:8.1f} {t_cv:8.1f} {t_gn + t_cv:8.1f} | {t_co:8.1f} {t_cg:8.1f} {t_co + t_cg:8.1f} | "
              f"{100 * (1 - (t_co + t_cg) / (t_gn + t_cv)):5.1f} %", flush=True)

if not args.no_ddim:
    from bench import LOW_GPU
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.model.unet_backbone import UNetDenoiser, build_unet_64x64
    from ddpm_diffusion_model_b200.testing.ddpim_inference import ddim_infer_sample
    torch.manual_seed(0)
    cfgs = [("low64", build_unet_64x64(**LOW_GPU), 64, B)]
    if args.c256:
        cfgs.append(("celeba256", UNetDenoiser(3, 128, (1, 1, 2, 2, 4), 2, {16}, 512, 0.0, 4, 64, 256), 256, 16))
    for name, model, S, n in cfgs:
        model = model.to(dev).eval()
        diff = Diffusion(T=1000, img_size=S).to(dev)
        res = {}
        for rnd in range(2):
            for flag in ("0", "1"):
                os.environ["DDPM_B200_FUSE_GN"] = flag

                def call():
                    with torch.autocast("cuda", dtype=torch.bfloat16), contextlib.redirect_stdout(io.StringIO()):
                        torch.manual_seed(5)
                        return ddim_infer_sample(model, diff, n=n, img_size=S, device="cuda:0", out_path="/tmp/gn_ab.png", steps=100, eta=0.0)
                g = call(); torch.cuda.synchronize(); t0 = time.perf_counter(); g = call(); torch.cuda.synchronize(); dt = time.perf_counter() - t0
                res[flag] = (dt, g)
                print(f"{name} DDIM-100 B={n} fuse_gn={flag}: {dt * 1e3:8.1f} ms  {n / dt:8.1f} samples/s  {dt / 99 * 1e3:6.2f} ms/eval", flush=True)
        d = (res["0"][1].float() - res["1"][1].float()).abs()
        print(f"{name}: final grids fused vs unfused: mean abs diff {float(d.mean()):.2e}, max {float(d.max()):.2e}", flush=True)
        os.environ.pop("DDPM_B200_FUSE_GN", None)
