"""Run-to-run determinism of one backward pass (diagnostic): same weights, same batch, same seeds, R repetitions;
reports which parameter gradients differ bitwise between repetitions and by how much relative to the gradient's
scale.  fp32 atomics (GroupNorm dgamma/dbeta, bias column sums) may reorder; tensor-core paths must not differ.
    python tools/determinism_check.py [tiny|low]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from bench import LOW_GPU
from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
from ddpm_diffusion_model_b200.model.unet_backbone import UNetDenoiser, build_unet_64x64

which = sys.argv[1] if len(sys.argv) > 1 else "tiny"
R = 6
dev = torch.device("cuda", 0)
torch.manual_seed(0)
if which == "tiny":
    model = UNetDenoiser(3, 32, (1, 2), 1, {8}, 64, 0.0, 2, 16, 16).to(dev).train(); B, S = 4, 16
else:
    model = build_unet_64x64(**LOW_GPU).to(dev).train(); B, S = 32, 64
diff = Diffusion(T=1000, img_size=S).to(dev)
x = torch.empty(B, 3, S, S, device=dev).uniform_(-1, 1)
names = [n for n, _ in model.named_parameters()]
runs = []
for r in range(R):
    for p in model.parameters():
        p.grad = None
    torch.manual_seed(5)
    t = diff.sample_timesteps(B, device=dev)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        loss = diff.loss_simple(model, x, t)
    (loss * 1024.0).backward()
    torch.cuda.synchronize()
    runs.append((float(loss), [p.grad.detach().clone() for p in model.parameters()]))
print(f"{which}: losses {[f'{l:.7f}' for l, _ in runs]}")
bad = {}
for r in range(1, R):
    for n, a, b in zip(names, runs[0][1], runs[r][1]):
        if not torch.equal(a, b):
            rel = float((a - b).abs().max() / a.abs().max().clamp_min(1e-30))
            bad[n] = max(bad.get(n, 0.0), rel)
print(f"{len(bad)} of {len(names)} parameter gradients differ between repetitions")
for n, rel in sorted(bad.items(), key=lambda kv: -kv[1])[:25]:
    print(f"   {n:50s} max|diff|/max|g| = {rel:.3e}")
