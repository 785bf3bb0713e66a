#!/usr/bin/env python
"""bench.py -- headline benchmark of the DDPM/DDIM hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload train|ddim] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[1]): CelebA64 low-GPU UNetDenoiser (12.68 M params), T=1000 linear
betas, bf16 autocast + GradScaler + AdamW(lr 2e-4) + EMA(0.9995) + grad-clip 1.0, batch 128 per GPU,
synthetic 64x64 images, data-parallel over N GPUs (weak scaling).  One "step" = one optimiser step.

  value    : images/s, whole job, batch already resident in HBM when the timed region starts; the K timed steps are
             ONE `train_one_epoch` call over a K-batch loader (the reference API's unit of work)
  e2e      : same metric through the public API with every batch in pinned HOST memory: per step the H2D copy of
             the images and a D2H DMA of the step's loss (pinned trace) inside the timing; `sync_every_step` is the
             same with one call per step (host reads the loss after every step)
  roofline : the dominant kernel (implicit-GEMM convolution) timed alone with CUDA events on the
             launching stream, algorithmic FLOPs / time vs the measured bf16 peak
  cpu_baseline / --impl reference : the UNMODIFIED reference (vendored byte-for-byte into git-ignored baseline/_ref by
             tools/vendor_reference.py) on the host cores through its own API -- train_one_epoch(device="cpu") at the
             arm's batch (B=128, bf16 CPU autocast = the function's default; fp32 beside it) and
             ddim_infer_sample(steps=100, n=8); that process never imports the product package
  gpu_eager_baseline : the same unmodified reference on the same B200 through PyTorch eager (cuDNN/cuBLAS/SDPA, bf16
             autocast + GradScaler + channels_last + cudnn.benchmark) in a subprocess -- the kernel-for-kernel bar
             (SURVEY.md section 2.2); `vs_gpu_eager` = ours / eager
  configs  : the 256-px half of the metric (BASELINE configs[2..4]): CelebA256 UNet train (B=32/GPU), DDIM-100 and
             DDPM-1000 sampling, batch-sharded over the ranks
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

LOW_GPU = dict(base_channels=96, channel_mults=(1, 2, 2, 2), num_res_blocks=1, attn_resolutions={8},
               num_heads=2, head_dim=32, dropout=0.1)
TRAIN_GF_PER_IMG = 47.94      # SURVEY.md §8d (fprop+dgrad+wgrad, measured on the reference with hooks)
FWD_GF_PER_IMG = 15.98


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sus=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sus=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], threading.Event()
        self.th = threading.Thread(target=self.run, daemon=True)

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.05)

    def __enter__(self):
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join(2)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = max([int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()] or [0])
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the UNMODIFIED reference (baseline/_ref) on the host cores.  Nothing here imports the
# product package or oracle/.
# ------------------------------------------------------------------------------------------------
def _ref_arm():
    import importlib.util
    spec = importlib.util.spec_from_file_location("_ddpm_reference_arm", os.path.join(ROOT, "baseline", "reference_arm.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return                                        # under torchrun only rank 0 times the host arm
    RA = _ref_arm()
    why = RA.available()
    if why:
        GUARD.emit(json.dumps({"impl": "reference", "unavailable": why}))
        return
    cores = RA.set_host_threads()                     # explicit: torchrun exports OMP_NUM_THREADS=1
    B = args.ref_batch
    steps = max(1, min(args.steps, args.ref_max_steps))
    warm = 1 if args.warmup else 0
    ips, sec, loss = RA.cpu_train(B, steps, warm, use_autocast=True)
    extra = {}
    if not args.ref_quick:
        ips32, sec32, _ = RA.cpu_train(min(B, 32), 1, 1, use_autocast=False)
        extra["train_fp32"] = {"value": ips32, "unit": "img/s", "ms_per_step": sec32 * 1e3,
                               "sample": f"1 optimiser step (after 1 warm-up) at B={min(B, 32)}, use_autocast=False"}
        sps, dt, evals = RA.cpu_ddim(args.ref_ddim_n, 100)
        extra["ddim100"] = {"value": sps, "unit": "samples/s", "steps": 100, "unet_evals": evals, "batch": args.ref_ddim_n, "img": 64,
                            "dtype": "f32", "seconds": dt, "timed": "whole ddim_infer_sample(device='cpu') call incl. grid PNG"}
    ddim_head = args.workload == "ddim" and "ddim100" in extra
    sample = (f"{steps} optimiser steps (after {warm} warm-up) of train_one_epoch(device='cpu', use_autocast=True -> CPU bf16 "
              f"autocast, the function's default) at B={B}, 64x64, dropout 0.1, AdamW+EMA+clip")
    line = {
        "impl": "reference",
        "metric": "ddim100_samples_per_s" if ddim_head else "train_img_per_s",
        "value": extra["ddim100"]["value"] if ddim_head else ips,
        "unit": "samples/s" if ddim_head else "img/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": (extra["ddim100"]["seconds"] / 99 if ddim_head else sec) * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32" if ddim_head else "bf16 (CPU autocast)",
        "data": "synthetic",
        "config": {"workload": "CelebA64 low-GPU UNet (12.68M) " + ("DDIM-100 sampling" if ddim_head else
                               "training step: bf16 autocast + AdamW + EMA + clip") + ", UNMODIFIED reference on host CPU",
                   "batch_per_gpu": args.ref_ddim_n if ddim_head else B, "img": 64, "T": 1000,
                   "reference_tree": RA.manifest_id(), "torch_threads": cores, "os_cpu_count": os.cpu_count()},
        "cpu_baseline": {"value": extra["ddim100"]["value"] if ddim_head else ips, "unit": "samples/s" if ddim_head else "img/s",
                         "cores": cores, "kind": "reference", "sample": "ddim_infer_sample(steps=100, n=%d)" % args.ref_ddim_n if ddim_head else sample},
        "e2e": {"value": extra["ddim100"]["value"] if ddim_head else ips, "unit": "samples/s" if ddim_head else "img/s",
                "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "loss": loss, **extra,
    }
    GUARD.emit(json.dumps(line))


def _json_subprocess(cmd, timeout):
    """Run a helper (reference arms) in its own process and parse the last JSON line of its stdout."""
    try:
        env = dict(os.environ)
        for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "OMP_NUM_THREADS"):
            env.pop(k, None)
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env, cwd=ROOT)
        for ln in reversed(out.stdout.strip().splitlines()):
            ln = ln.strip()
            if ln.startswith("{"):
                return json.loads(ln)
        return {"unavailable": f"no JSON from {' '.join(cmd[-4:])} (rc {out.returncode}): {out.stderr[-200:]}"}
    except Exception as ex:                           # noqa: BLE001
        return {"unavailable": f"{type(ex).__name__}: {ex}"[:300]}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
C256_SHAPES = [(128, 128, 256, 10), (128, 128, 128, 9), (256, 256, 64, 9), (256, 128, 256, 1), (256, 256, 128, 1),
               (512, 512, 16, 12), (384, 128, 128, 1), (256, 256, 32, 9), (512, 256, 64, 1)]     # SURVEY.md Appendix A.2


def conv_roofline(device, batch, reps=5, shapes=None):
    """Time the implicit-GEMM convolution kernel alone (fprop shapes of the low-GPU UNet at the bench
    batch), CUDA events on the launching stream.  Returns (flops per pass, seconds per pass, detail)."""
    from ddpm_diffusion_model_b200 import _lib, engine
    E = engine.Exec(device, _lib.BF16, False, False)
    # (Cin, Cout, H, count) -- SURVEY.md Appendix A.1, 3x3 s1 rows that make up 90 % of the FLOPs
    if shapes is None:
        shapes = [(96, 96, 64, 5), (192, 192, 32, 5), (192, 192, 64, 1), (288, 96, 64, 1), (384, 192, 32, 1),
                  (192, 192, 16, 6), (192, 192, 8, 9), (96, 192, 32, 1), (384, 192, 16, 1)]
    tot_f, tot_t, detail = 0.0, 0.0, []
    for ci, co, hw, cnt in shapes:
        w = torch.nn.Parameter(torch.randn(co, ci, 3, 3, device=device) * 0.02)
        wf, _ = E.wcache.get(E, w, _lib.BF16, False)
        x = E.act(batch, hw, hw, ci)
        x.interior().normal_()
        y = E.act(batch, hw, hw, co)
        engine.conv(E, x, wf, y, 3, 1, 1)
        torch.cuda.synchronize(device)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(reps):
            engine.conv(E, x, wf, y, 3, 1, 1)
        e.record()
        torch.cuda.synchronize(device)
        dt = s.elapsed_time(e) / 1e3 / reps
        fl = 2.0 * batch * hw * hw * co * ci * 9
        detail.append({"shape": f"{ci}->{co}@{hw}", "tflops": fl / dt / 1e12, "us": dt * 1e6})
        tot_f += fl * cnt
        tot_t += dt * cnt
        del x, y
    return tot_f, tot_t, detail


def _build_ours(config, dev):
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.model.unet_backbone import UNetDenoiser, build_unet_64x64
    from ddpm_diffusion_model_b200.training_loops.ema import EMA
    from ddpm_diffusion_model_b200.training_loops.grad_scaler import make_grad_scaler
    torch.manual_seed(0)
    if config == "celeba256":
        # BASELINE.json configs[2]: CelebA256 attention UNet (63.1 M params), bf16, batch 32 per GPU
        model = UNetDenoiser(3, 128, (1, 1, 2, 2, 4), 2, {16}, 512, 0.1, 4, 64, 256).to(dev)
        opt = torch.optim.AdamW(model.parameters(), lr=2e-4, betas=(0.9, 0.999), weight_decay=0.005)
        ema_decay, gf_train, img = 0.9997, 1257.3, 256
    else:
        model = build_unet_64x64(**LOW_GPU).to(dev)
        opt = torch.optim.AdamW(model.parameters(), lr=2e-4, betas=(0.9, 0.999), weight_decay=0.0)
        ema_decay, gf_train, img = 0.9995, TRAIN_GF_PER_IMG, 64
    diff = Diffusion(T=1000, schedule="linear", beta_min=1e-4, beta_max=2e-2, img_size=img).to(dev)
    return model, diff, opt, EMA(model, decay=ema_decay), make_grad_scaler("cuda", True), gf_train, img


DUMP_SAMPLE = 1 << 21          # elements kept per parameter-sized array: 8 MB each in float32, 32 MB for all four


def dump_outputs(out_dir, model, opt, ema, scaler, ret, losses):
    """Write what the timed `train_one_epoch` call hands back to its caller, as .npy files: its return value, the per-step
    losses, and the model state the last step left behind (parameters, AdamW moments, EMA shadow; flattened in
    `model.parameters()` order and sampled at the same fixed, seeded indices, sorted).  The gradients are not written:
    the step zeroes them."""
    import numpy as np
    params = list(model.parameters())
    n = sum(p.numel() for p in params)
    idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values

    def sampled(ts):
        return torch.cat([t.detach().reshape(-1).cpu() for t in ts])[idx].numpy().astype(np.float32)

    os.makedirs(out_dir, exist_ok=True)
    arrays = {
        "avg_loss": np.array([ret[0]], dtype=np.float64),
        "step_losses": losses.numpy().astype(np.float32),
        "grad_scale": np.array([scaler.get_scale()], dtype=np.float64),
        "params": sampled(params),
        "adam_exp_avg": sampled([opt.state[p]["exp_avg"] for p in params]),
        "adam_exp_avg_sq": sampled([opt.state[p]["exp_avg_sq"] for p in params]),
        "ema_shadow": sampled(ema.shadow),
    }
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args):
    import contextlib
    import io
    import tempfile
    import torch.distributed as dist
    from ddpm_diffusion_model_b200 import _lib
    from ddpm_diffusion_model_b200 import engine as _engine
    from ddpm_diffusion_model_b200.training_loops.train_one_epoch import last_enqueue_ms_per_step, last_graph_steps, last_step_losses, train_one_epoch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.tc_exp:
        _lib.lib.ddpm_set_tc_mode(1 | (args.tc_exp << 4), 0)
    c256 = args.config == "celeba256"
    B = 32 if (c256 and args.batch == 128) else args.batch
    model, diff, opt, ema, scaler, gf_train, IMG = _build_ours(args.config, dev)
    if c256:
        args.no_ddim = True
    torch.manual_seed(7 + rank)
    x_host = torch.empty(B, 3, IMG, IMG).uniform_(-1, 1).pin_memory()
    y_host = torch.zeros(B)
    x_dev = x_host.to(dev)
    kw = dict(scaler=scaler, ema=ema, device=f"cuda:{local}", grad_clip=1.0)

    # One `train_one_epoch` call over a K-batch loader is the reference API's unit of work (train_one_epoch.py:11);
    # inside it nothing synchronises with the host until the epoch's mean loss is read, so the enqueue of step i+1
    # overlaps the GPU work of step i.  (One call PER step drains the GPU at every call boundary; reported below as
    # `sync_every_step`.)
    def step_resident(K=1):
        return train_one_epoch(model, diff, [(x_dev, y_host)] * K, opt, **kw)

    # e2e: every step copies its batch from pinned host memory (the reference's x.to(device, non_blocking=True),
    # train_one_epoch.py:62; our loop issues the copy of batch i+1 on a copy stream while step i runs) and DMAs its 4-byte
    # loss back into a pinned trace (`last_step_losses()`).  All K copies happen inside the timed region.
    def step_e2e(K=1):
        return train_one_epoch(model, diff, [(x_host, y_host)] * K, opt, **kw)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(v):
        if world > 1:
            tt = torch.tensor([v], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt)
        return v

    def timed(fn, K, per_call=False):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        _lib.launch_count(reset=True)
        t0 = time.perf_counter()
        s.record()
        last = None
        if per_call:
            for _ in range(K):
                last = fn()
        else:
            last = fn(K)
        e.record()
        host_s = time.perf_counter() - t0              # host time to ENQUEUE the K steps (+ the final loss read)
        barrier()
        ms = s.elapsed_time(e)
        n_launch = _lib.launch_count(reset=True)
        return max_over_ranks(ms) / 1e3, n_launch, last, host_s

    if args.profile:                                  # short run for `ncu` launch lists
        for _ in range(2):
            step_resident()
        torch.cuda.synchronize(dev)
        torch.cuda.nvtx.range_push("timed_step")
        step_resident()
        torch.cuda.synchronize(dev)
        torch.cuda.nvtx.range_pop()
        return
    step_resident(max(3, args.warmup))
    miss0 = _engine.POOL.misses
    with ClockSampler(local) as clk:
        sec, launches, last, host_s = timed(step_resident, args.steps)
    enqueue_ms = last_enqueue_ms_per_step()           # host loop time per step, excluding the final synchronising loss read
    graph_steps = last_graph_steps()                  # timed steps that ran as ONE CUDA-graph replay each (train_one_epoch._GraphStep)
    pool_misses = _engine.POOL.misses - miss0
    if args.dump_outputs and rank == 0:               # before the legs below train the same model further
        dump_outputs(args.dump_outputs, model, opt, ema, scaler, last, last_step_losses())
    # ... which includes back-pressure once the launch queue is full (the GPU is the bottleneck at this batch).  The host's own
    # cost per step is what the same loop takes when the GPU is NOT the limit: the same epoch on two-image batches.
    x_tiny = x_dev[:2].contiguous()
    train_one_epoch(model, diff, [(x_tiny, y_host[:2])] * 3, opt, **kw)
    train_one_epoch(model, diff, [(x_tiny, y_host[:2])] * 8, opt, **kw)
    enqueue_unloaded_ms = last_enqueue_ms_per_step()
    step_e2e(2)
    sec_e2e, _, last_e2e, _ = timed(step_e2e, args.steps)
    trace = last_step_losses()
    assert trace.numel() == args.steps and bool(torch.isfinite(trace).all()), "per-step loss trace incomplete"
    sec_sync, _, _, _ = timed(step_e2e, min(args.steps, 20), per_call=True)
    sec_sync /= min(args.steps, 20)
    value = world * B * args.steps / sec
    e2e = world * B * args.steps / sec_e2e
    # input side (SURVEY 8(f) f4): the same epoch fed by the device-resident loader -- a uint8 dataset in HBM, per step one
    # gather + ToTensor + Normalize kernel instead of a host batch (what a real run uses at this rate)
    from ddpm_diffusion_model_b200.data import DeviceLoader
    u8 = torch.randint(0, 256, (B * args.steps, IMG, IMG, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(3 + rank))
    feeder = DeviceLoader(u8, B, shuffle=True, drop_last=True, device=dev, generator=torch.Generator().manual_seed(5), shard=False)
    sec_feed, _, _, _ = timed(lambda K: train_one_epoch(model, diff, feeder, opt, **kw), args.steps)
    del feeder, u8

    def sampler_leg(mdl, dff, kind, nb, img, steps):
        """Whole public sampler call (bf16 autocast, eta = 0, batch-sharded over ranks with no communication; includes
        the grid PNG write of the reference API).  Wall clock, barrier + synchronize on both sides, max over ranks."""
        from ddpm_diffusion_model_b200.testing.ddpim_inference import ddim_infer_sample
        from ddpm_diffusion_model_b200.testing.ddpm_inference import ddpm_infer_sample
        outp = os.path.join(tempfile.gettempdir(), f"{kind}_bench_{rank}.png")

        def call(n_steps):
            with torch.autocast("cuda", dtype=torch.bfloat16):
                if kind == "ddim":
                    ddim_infer_sample(mdl, dff, n=nb * world, img_size=img, device=f"cuda:{local}", ema=None, out_path=outp,
                                      seed=1234, steps=n_steps, eta=0.0, shard=world > 1)
                else:
                    ddpm_infer_sample(mdl, dff, n=nb * world, img_size=img, device=f"cuda:{local}", ema=None, out_path=outp,
                                      seed=1234, shard=world > 1)
        with contextlib.redirect_stdout(io.StringIO()):
            if kind == "ddim":
                call(min(steps, 12))                              # warm-up: pools / packed weights / schedule handle
            barrier()
            t0 = time.perf_counter()
            call(steps)
            barrier()
            dt = max_over_ranks(time.perf_counter() - t0)
        evals = steps - 1 if kind == "ddim" else dff.T
        mdl.train()
        return {"value": nb * world / dt, "unit": "samples/s", "steps": steps if kind == "ddim" else dff.T, "unet_evals": evals,
                "batch_per_gpu": nb, "img": img, "dtype": "bf16 autocast", "ms_per_eval": dt / evals * 1e3, "seconds": dt,
                "cuda_graph": os.environ.get("DDPM_B200_GRAPHS", "0") == "1",
                "timed": "whole %s_infer_sample call (wall clock, barrier + synchronize both sides), incl. grid PNG" % kind}

    # ---- second half of the metric: DDIM-100 samples/s through the public sampler
    ddim = None if args.no_ddim else sampler_leg(model, diff, "ddim", args.ddim_batch, IMG, 100)

    roof = cpu = eager = None
    if rank == 0:
        pk = peaks()
        fl, tt, detail = conv_roofline(dev, B, shapes=C256_SHAPES if c256 else None)
        ach = fl / tt / 1e12
        # traffic: dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of this kernel at the 96->96@64 shape
        # (B=128), from the committed `ncu --set full` capture profiles/r2_ncu_prof_conv_96_96_64.txt
        # (107.3 MB read = the input tensor once, 63.9 MB written back before the kernel ended; the algorithmic
        # bytes of that launch are 107 MB in + 107 MB out + 0.17 MB weights)
        roof = {"bound": "tensor", "achieved": ach, "peak": pk["tf_burst"], "unit": "TFLOP/s", "frac": ach / pk["tf_burst"],
                "traffic": 171145216 if (B == 128 and not c256) else None, "traffic_shape": "96->96@64, B=128",
                "kernel": "conv_tc2_kernel (tcgen05 cta_group::2 implicit GEMM; 3x3 s1 layers of the %s UNet, count-weighted, B=%d)" % ("CelebA256" if c256 else "low-GPU", B),
                "peak_source": pk["src"] + " bf16 burst (kernel timed alone)", "per_shape": detail,
                "step_tensor_frac": (gf_train * 1e9 * world * B * args.steps / sec) / (world * pk["tf_sus"] * 1e12)}

    # ---- the 256-px half of the metric (BASELINE configs[2..4]); the 64-px model and its buffers are released first
    configs = None
    if not c256 and not args.no_c256:
        del model, diff, opt, ema, scaler, kw
        _engine.POOL.clear()
        torch.cuda.empty_cache()
        m2, d2, o2, e2, s2, gf2, _ = _build_ours("celeba256", dev)
        B2 = args.c256_batch
        torch.manual_seed(11 + rank)
        x2 = torch.empty(B2, 3, 256, 256).uniform_(-1, 1).pin_memory()
        y2 = torch.zeros(B2)
        kw2 = dict(scaler=s2, ema=e2, device=f"cuda:{local}", grad_clip=1.0)
        K2 = max(3, min(args.steps, args.c256_steps))
        train_one_epoch(m2, d2, [(x2, y2)] * 3, o2, **kw2)
        sec2, launches2, last2, _ = timed(lambda K: train_one_epoch(m2, d2, [(x2, y2)] * K, o2, **kw2), K2)
        configs = {"celeba256_train": {
            "metric": "train_img_per_s", "value": world * B2 * K2 / sec2, "unit": "img/s", "ms_per_step": sec2 / K2 * 1e3, "steps": K2,
            "batch_per_gpu": B2, "img": 256, "params": 63100675, "dtype": "bf16", "gpu_launches": launches2, "loss": last2[0],
            "train_tflops_per_gpu": gf2 * 1e9 * B2 * K2 / sec2 / 1e12,
            "step_tensor_frac": (gf2 * 1e9 * B2 * K2 / sec2) / (peaks()["tf_sus"] * 1e12),
            "timed": "one train_one_epoch call over K pinned HOST batches (H2D of the batch + D2H of the loss every step), CUDA events, max over ranks"}}
        del o2, e2, s2, kw2, x2
        m2.zero_grad(set_to_none=True)
        _engine.POOL.clear()
        torch.cuda.empty_cache()
        configs["celeba256_ddim100"] = sampler_leg(m2, d2, "ddim", args.c256_ddim_batch, 256, 100)
        if not args.no_ddpm:
            _engine.POOL.clear()
            torch.cuda.empty_cache()
            configs["celeba256_ddpm1000"] = sampler_leg(m2, d2, "ddpm", args.c256_ddpm_batch, 256, 1000)
        del m2, d2
        _engine.POOL.clear()
        torch.cuda.empty_cache()

    if rank == 0 and world == 1:
        py = sys.executable
        if not args.no_cpu:
            # bounded sample of the UNMODIFIED reference on this box's host cores (own process: no product code mapped)
            r = _json_subprocess([py, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                                  "--ref-quick", "--ref-batch", "32"], 600)
            cpu = r.get("cpu_baseline") if "cpu_baseline" in r else {"value": None, "unit": "img/s", "cores": None, "kind": "reference",
                                                                       "sample": r.get("unavailable", "failed")}
        if not args.no_eager:
            # the same unmodified reference on THIS B200 through PyTorch eager -- the kernel-for-kernel bar
            eager = {"low64": _json_subprocess([py, os.path.join(ROOT, "baseline", "reference_arm.py"), "gpu", "low64", str(B),
                                                 str(min(args.steps, 10)), str(0 if args.no_ddim else args.ddim_batch), "100"], 900)}
            if configs is not None:
                eager["celeba256"] = _json_subprocess([py, os.path.join(ROOT, "baseline", "reference_arm.py"), "gpu", "celeba256",
                                                       str(args.c256_batch), "5", str(args.c256_ddim_batch), "100"], 900)
    if rank == 0:
        vs_eager = None
        if eager:
            vs_eager = {}
            lo = eager.get("low64", {})
            if "train" in lo:
                vs_eager["train_e2e"] = e2e / lo["train"]["value"]
                vs_eager["train_device"] = value / lo["train"]["value"]
            if ddim and "ddim" in lo:
                vs_eager["ddim100"] = ddim["value"] / lo["ddim"]["value"]
            hi = eager.get("celeba256", {})
            if configs and "train" in hi:
                vs_eager["celeba256_train"] = configs["celeba256_train"]["value"] / hi["train"]["value"]
            if configs and "ddim" in hi:
                vs_eager["celeba256_ddim100"] = configs["celeba256_ddim100"]["value"] / hi["ddim"]["value"]
        line = {
            "metric": "train_img_per_s", "value": value, "unit": "img/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": sec / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": ("CelebA256 attention UNet (63.1M)" if c256 else "CelebA64 low-GPU UNet (12.68M)") +
                       " training step: bf16 autocast + GradScaler + AdamW + EMA + clip",
                       "batch_per_gpu": B, "global_batch": B * world, "img": IMG, "T": 1000, "parallelism": f"dp{world}",
                       "timed": "one train_one_epoch call over K batches",
                       "l2": "working set per step (~3 GB of activations) exceeds the 126 MB L2; no explicit flush"},
            "e2e": {"value": e2e, "unit": "img/s", "h2d_bytes_per_step": B * 3 * IMG * IMG * 4, "d2h_bytes_per_step": 4,
                    "ms_per_step": sec_e2e / args.steps * 1e3,
                    "timed": "one train_one_epoch call over K pinned host batches, all inside the timed region: H2D of every batch (copy stream, one "
                             "step ahead); every step's loss DMA'd to the pinned trace (eager steps: 4 B per step as they finish; CUDA-graph "
                             "steps: from the device ring in one copy when the epoch ends); one synchronising read of the mean loss at the end",
                    "device_feeder": {"value": world * B * args.steps / sec_feed, "ms_per_step": sec_feed / args.steps * 1e3,
                                      "timed": "same epoch fed by DeviceLoader (uint8 dataset resident in HBM, shuffled; one "
                                               "gather+ToTensor+Normalize kernel per step)"},
                    "sync_every_step": {"value": world * B / sec_sync, "ms_per_step": sec_sync * 1e3,
                                        "timed": "one train_one_epoch call PER step (host reads the loss after every step)"}},
            "gpu_launches": launches, "cuda_graph_steps": graph_steps, "host_enqueue_ms_per_step": enqueue_ms, "host_enqueue_ms_per_step_unloaded": enqueue_unloaded_ms,
            "clocks": clk.summary(), "roofline": roof, "cpu_baseline": cpu,
            "loss": last[0] if last else None, "pool_misses_in_timed_region": pool_misses, "ddim100": ddim,
            "train_tflops_per_gpu": gf_train * 1e9 * B * args.steps / sec / 1e12,
            "configs": configs, "gpu_eager_baseline": eager, "vs_gpu_eager": vs_eager,
        }
        GUARD.emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


class _StdoutGuard:
    """Everything written to fd 1 while the benchmark runs (NCCL's version banner, sampler progress prints, library
    chatter) goes to stderr; only `emit()` reaches the real stdout -> exactly ONE JSON line."""

    def __init__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, line: str):
        sys.stdout.flush()
        os.write(self.real, (line + "\n").encode())


GUARD = None


def main():
    global GUARD
    if os.environ.get("DDPM_BENCH_WATCHDOG"):            # diagnostics: dump every thread's Python stack if the run stalls
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ["DDPM_BENCH_WATCHDOG"]), repeat=True, file=sys.stderr)
    GUARD = _StdoutGuard()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="train", choices=["train", "ddim"],
                    help="--impl reference: which half of the metric is the line's headline value (the other is a field)")
    ap.add_argument("--ref-batch", type=int, default=128, help="--impl reference: batch of the host train step (the arm's B)")
    ap.add_argument("--ref-max-steps", type=int, default=3, help="--impl reference: cap on timed host steps (bounded sample)")
    ap.add_argument("--ref-ddim-n", type=int, default=8, help="--impl reference: images of the host DDIM-100 leg")
    ap.add_argument("--ref-quick", action="store_true", help="--impl reference: bf16 train leg only (cpu_baseline of our line)")
    ap.add_argument("--no-eager", action="store_true", help="skip the gpu_eager_baseline legs (reference on this B200, PyTorch eager)")
    ap.add_argument("--no-c256", action="store_true", help="skip the 256-px block (CelebA256 train / DDIM-100 / DDPM-1000)")
    ap.add_argument("--no-ddpm", action="store_true", help="skip DDPM-1000 @256 (the longest leg, ~45 s)")
    ap.add_argument("--c256-batch", type=int, default=32)
    ap.add_argument("--c256-steps", type=int, default=8)
    ap.add_argument("--c256-ddim-batch", type=int, default=16)
    ap.add_argument("--c256-ddpm-batch", type=int, default=64)
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--config", default="low64", choices=["low64", "celeba256"],
                    help="low64: BASELINE configs[1] (default, the metric's workload); celeba256: configs[2] (batch 32/GPU)")
    ap.add_argument("--tc-exp", type=int, default=0, help="diagnostic flags for the conv kernel (timing experiments only; results are wrong)")
    ap.add_argument("--no-ddim", action="store_true", help="skip the DDIM-100 sampling leg")
    ap.add_argument("--ddim-batch", type=int, default=256, help="images per GPU for the DDIM-100 leg")
    ap.add_argument("--profile", action="store_true", help="2 warm-up steps + 1 step, no JSON (for ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed train_one_epoch call returned and left in the model after its last step "
                         "to DIR/<name>.npy (float32/float64, 32 MB; large arrays as a fixed seeded sample); same "
                         "arguments give the same inputs, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.profile):
        ap.error("--dump-outputs needs --impl ours and no --profile")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
