"""Per-kernel roofline table on the GPU (run under gpurun).

Times every kernel family of the hot path alone, at the shapes of the bench workload (low-GPU UNet,
B=128 by default), with CUDA events on the launching stream, and prints achieved TFLOP/s or GB/s
against MEASURED_PEAKS.json.  Algorithmic bytes / FLOPs per launch are the DESIGN.md figures.

    python tools/kbench.py [--batch 128] [--only conv,wgrad,gn,colsum,ew,param] [--tcexp FLAGS] [--json out.json]
"""
import argparse, json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from ddpm_diffusion_model_b200 import _lib, engine

ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=128)
ap.add_argument("--only", default="conv,wgrad,gn,colsum,ew,param")
ap.add_argument("--reps", type=int, default=10)
ap.add_argument("--json", default=None)
ap.add_argument("--epi", action="store_true", help="conv: also time with bias + time-bias + residual epilogue")
ap.add_argument("--gnshape", default=None, help="restrict gn to one 'C,H'")
ap.add_argument("--tcexp", type=int, default=0, help="path-forcing flags for the whole run (ddpm_set_tc_mode(1 | flags << 4)): 32 = conv channel tiles wider than 128, 64 = conv weights streamed instead of resident, 128 = no 32-byte conv epilogue stores, 1024 = single-CTA wgrad kernel instead of the pair kernel")
ap.add_argument("--shape", default=None, help="restrict conv/wgrad to one 'Cin,Cout,H' (for ncu)")
args = ap.parse_args()
only = set(args.only.split(","))
dev = torch.device("cuda", 0)
B = args.batch
pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}
HBM, TF = pk["hbm_gbs"], pk["bf16_tflops"]
flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
rows = []


def timeit(fn, reps=None, flush=False):
    reps = reps or args.reps
    fn(); fn()
    torch.cuda.synchronize()
    if flush:                                   # cold-L2 timing: flush before every rep, time each rep alone
        tot = 0.0
        for _ in range(reps):
            flush_buf.zero_()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record(); fn(); e.record()
            torch.cuda.synchronize()
            tot += s.elapsed_time(e)
        return tot / reps * 1e-3
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / reps * 1e-3


def report(kind, name, sec, flops=None, nbytes=None, cnt=1):
    r = {"kind": kind, "name": name, "us": sec * 1e6, "count_per_step": cnt}
    if flops is not None:
        r["tflops"] = flops / sec / 1e12; r["frac"] = r["tflops"] / TF
        print(f"{kind:8s} {name:28s} {sec*1e6:9.1f} us  {r['tflops']:8.1f} TFLOP/s  {100*r['frac']:5.1f}% of bf16 burst  x{cnt}", flush=True)
    else:
        r["gbs"] = nbytes / sec / 1e9; r["frac"] = r["gbs"] / HBM
        print(f"{kind:8s} {name:28s} {sec*1e6:9.1f} us  {r['gbs']:8.1f} GB/s     {100*r['frac']:5.1f}% of HBM copy   x{cnt}", flush=True)
    rows.append(r)


# (Cin, Cout, H, count fwd) -- SURVEY.md Appendix A.1
CONV = [(96, 96, 64, 5), (192, 192, 32, 5), (192, 192, 64, 1), (288, 96, 64, 1), (384, 192, 32, 1),
        (192, 192, 16, 6), (192, 192, 8, 9), (96, 192, 32, 1), (384, 192, 16, 1), (384, 192, 8, 1)]
if args.shape:
    CONV = []
    for sh in args.shape.split(";"):
        v = [int(t) for t in sh.split(",")]
        CONV.append((v[0], v[1], v[2], 1) + ((v[3],) if len(v) > 3 else ()))
GN = [(96, 64, 6), (96, 32, 1), (192, 32, 4), (192, 16, 5), (192, 8, 11), (384, 8, 1), (384, 16, 1), (384, 32, 1), (288, 64, 1)]

if args.gnshape:
    c_, h_ = [int(v) for v in args.gnshape.split(",")]
    GN = [(c_, h_, 1)]
E = engine.Exec(dev, _lib.BF16, True, True, rng=torch.tensor([1, 0], dtype=torch.int64, device=dev))
_lib.call("ddpm_set_tc_mode", 1 | (args.tcexp << 4), 0)

if "conv" in only:
    for ci, co, hw, cnt, *kk in CONV:
        ks = kk[0] if kk else 3
        w = torch.nn.Parameter(torch.randn(co, ci, ks, ks, device=dev) * 0.02)
        wf, _ = E.wcache.get(E, w, _lib.BF16, False)
        x = E.act(B, hw, hw, ci); x.interior().normal_()
        y = E.act(B, hw, hw, co)
        fl = 2.0 * B * hw * hw * co * ci * ks * ks
        sec = timeit(lambda: engine.conv(E, x, wf, y, ks, 1, ks // 2))
        report("conv", f"{ci}->{co}@{hw}k{ks}", sec, flops=fl, cnt=2 * cnt)
        if args.epi:
            bias = torch.randn(co, device=dev); tb = torch.randn(B, co, device=dev)
            r = E.act(B, hw, hw, co); r.interior().normal_()
            sec = timeit(lambda: engine.conv(E, x, wf, y, ks, 1, ks // 2, bias=bias, tbias=tb, res=r))
            report("conv", f"{ci}->{co}@{hw}k{ks} skip(+bias+tbias+res)", sec, flops=fl, cnt=2 * cnt)
            sec = timeit(lambda: engine.conv(E, x, wf, y, ks, 1, ks // 2, bias=bias, accum=True))
            report("conv", f"{ci}->{co}@{hw}k{ks} skip(+bias+accum)", sec, flops=fl, cnt=2 * cnt)
            del r
        del x, y

if "wgrad" in only:
    for ci, co, hw, cnt, *kk in CONV:
        w = torch.nn.Parameter(torch.zeros(co, ci, 3, 3, device=dev))
        x = E.act(B, hw, hw, ci); x.interior().normal_()
        dy = E.act(B, hw, hw, co); dy.interior().normal_()
        fl = 2.0 * B * hw * hw * co * ci * 9
        sec = timeit(lambda: engine.wgrad(E, x, dy, w, 3, 1, 1))
        report("wgrad", f"{ci}->{co}@{hw}", sec, flops=fl, cnt=cnt)
        bpar = torch.nn.Parameter(torch.zeros(co, device=dev))
        sec = timeit(lambda: engine.wgrad(E, x, dy, w, 3, 1, 1, bias=bpar))
        report("wgrad", f"{ci}->{co}@{hw} skip(+bias grad)", sec, flops=fl, cnt=cnt)
        del x, dy

if "gn" in only:
    for c, hw, cnt in GN:
        gn = torch.nn.GroupNorm(32, c, eps=1e-6).to(dev)
        x = E.act(B, hw, hw, c); x.interior().normal_()
        o = E.act(B, hw, hw, c)
        dy = E.act(B, hw, hw, c); dy.interior().normal_()
        dx = E.act(B, hw, hw, c)
        n = B * hw * hw * c
        fl = n * 2 > (100 << 20)            # flush L2 between reps only when the tensor would not fit anyway
        st = engine.gn_stats(E, x, 32)
        report("gn", f"stats {c}@{hw}", timeit(lambda: engine.gn_stats(E, x, 32), flush=fl), nbytes=2 * n, cnt=cnt)
        report("gn", f"apply+silu {c}@{hw}", timeit(lambda: engine.gn_apply(E, x, st, gn, 1, 0.0, 0, out=o), flush=fl), nbytes=4 * n, cnt=cnt)
        report("gn", f"FUSED fwd silu+drop {c}@{hw}", timeit(lambda: engine.gn_fwd(E, x, gn, 1, 0.1, 3, out=o), flush=fl), nbytes=4 * n, cnt=cnt)
        report("gn", f"apply+silu+drop {c}@{hw}", timeit(lambda: engine.gn_apply(E, x, st, gn, 1, 0.1, 3, out=o), flush=fl), nbytes=4 * n, cnt=cnt)
        report("gn", f"bwd(silu+drop) {c}@{hw}", timeit(lambda: engine.gn_bwd(E, x, st, gn, 1, 0.1, 3, dy, dx, False, dy_scratch=True), flush=fl), nbytes=6 * n, cnt=cnt)
        report("gn", f"skip bwd accumulate {c}@{hw}", timeit(lambda: engine.gn_bwd(E, x, st, gn, 1, 0.0, 0, dy, dx, True, dy_scratch=True), flush=fl), nbytes=8 * n, cnt=cnt)
        report("gn", f"skip FUSED fwd silu (eval) {c}@{hw}", timeit(lambda: engine.gn_fwd(E, x, gn, 1, 0.0, 0, out=o), flush=fl), nbytes=4 * n, cnt=cnt)
        del x, o, dy, dx

if "colsum" in only:
    for c, hw, cnt in [(96, 64, 12), (192, 32, 12), (192, 16, 12), (192, 8, 20)]:
        dy = E.act(B, hw, hw, c); dy.interior().normal_()
        out = torch.empty(B, c, device=dev)
        bias = torch.nn.Parameter(torch.zeros(c, device=dev))
        report("colsum", f"{c}@{hw}", timeit(lambda: engine.colsum(E, dy, out, bias)), nbytes=2 * B * hw * hw * c, cnt=cnt)
        del dy

if "ew" in only:
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion, to_image01
    diff = Diffusion(T=1000).to(dev)
    for (b, s) in [(B, 64), (64, 256), (160, 256)]:       # 160 x 3 x 256 x 256: 126 MB per fp32 tensor, 380-500 MB working sets (> L2, SURVEY 8d)
        x0 = torch.randn(b, 3, s, s, device=dev); eps = torch.randn_like(x0); z = torch.randn_like(x0)
        t = torch.randint(1, 1000, (b,), device=dev); tp = (t - 10).clamp(min=0)
        n = x0.numel()
        report("ew", f"q_sample B{b}@{s}", timeit(lambda: diff.q_sample(x0, t, eps)), nbytes=12 * n)
        report("ew", f"ddpm_step B{b}@{s}", timeit(lambda: diff.p_sample_step(lambda a, b_: eps, x0, t, noise=z)), nbytes=16 * n)
        report("ew", f"ddim_step eta0 B{b}@{s}", timeit(lambda: diff.p_sample_step_ddim(lambda a, b_: eps, x0, t, tp, eta=0.0, noise=z)), nbytes=12 * n)
        report("ew", f"ddim_step eta1 B{b}@{s}", timeit(lambda: diff.p_sample_step_ddim(lambda a, b_: eps, x0, t, tp, eta=1.0, noise=z)), nbytes=16 * n)
        report("ew", f"to_image01 B{b}@{s}", timeit(lambda: to_image01(x0)), nbytes=8 * n)

if "param" in only:
    for n in (12_680_259, 63_100_675):
        p, g, m, v, ema = (torch.randn(n, device=dev) * 0.01 for _ in range(5))
        v.abs_()
        stats = torch.zeros(4, dtype=torch.float32, device=dev)
        scale = torch.ones(1, device=dev); step = torch.ones(1, dtype=torch.float32, device=dev)
        try:
            import ctypes as C
            hy = _lib.AdamHyper(2e-4, 0.9, 0.999, 1e-8, 0.0, 1.0, 0.9995, 1)
            def upd():
                _lib.call("ddpm_param_reduce", g.data_ptr(), n, stats.data_ptr(), E.stream)
                _lib.call("ddpm_param_update", p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), ema.data_ptr(), n,
                          stats.data_ptr(), step.data_ptr(), scale.data_ptr(), C.byref(hy), E.stream)
            report("param", f"reduce+update n={n}", timeit(upd, flush=True), nbytes=40 * n)
        except Exception as ex:                       # signature drift: report, do not hide
            print("param bench failed:", ex)

if args.json:
    json.dump({"batch": B, "peaks": pk, "rows": rows}, open(args.json, "w"), indent=1)
# per-step totals (count_per_step x time) so shares can be compared with the ncu launch list
tot = {}
for r in rows:
    if " skip" in r["name"] or (r["kind"] == "gn" and not (r["name"].startswith("FUSED") or r["name"].startswith("bwd"))):
        continue
    tot[r["kind"]] = tot.get(r["kind"], 0.0) + r["us"] * r["count_per_step"]
print({k: round(v / 1e3, 3) for k, v in tot.items()}, "ms per train step (kernel families, timed alone)")
