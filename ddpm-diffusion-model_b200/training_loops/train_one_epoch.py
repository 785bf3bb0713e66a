"""Drop-in for src/training_loops/train_one_epoch.py (same signature and return value).

What changes underneath (SURVEY.md §3.1): the UNet fwd/bwd run on libddpm_b200; parameters live in a
flat arena; `scaler.unscale_ + clip_grad_norm_ + optimizer.step + scaler.update + ema.update`
collapse into one reduction + one fused update kernel when the optimiser is torch Adam/AdamW; the
per-micro-batch `float(loss)` host sync (train_one_epoch.py:119) becomes a device-side sum read once
at the end; under torch.distributed the gradient arena is averaged bucket by bucket during backward.
"""
import ctypes as C
import os
import time

import torch

from .. import _lib
from .. import dist as _dist
from ..arena import ensure_arena
from ..engine import GLOBAL_WCACHE, GRAPH_EPOCH, POOL
from .ema import EMA  # noqa: F401
from .grad_scaler import autocast_ctx, make_grad_scaler  # noqa: F401
from .training_utils import compute_grad_norm, gpu_mem_mb


def _stream(dev) -> int:
    return _lib.stream_for(dev)


class _LossTrace:
    """Per-step losses of the last epoch without a per-step host sync: every step DMAs its 4-byte loss into a pinned
    host chunk (non-blocking); the values are valid once `train_one_epoch` has returned (it ends with one
    synchronising read of the device-side sum).  `last_step_losses()` returns them as a CPU tensor."""
    CHUNK = 1024

    def __init__(self):
        self.chunks, self.n = [], 0

    def reset(self):
        self.n = 0

    def push(self, loss: torch.Tensor):
        c, k = divmod(self.n, self.CHUNK)
        if c == len(self.chunks):
            self.chunks.append(torch.empty(self.CHUNK, dtype=torch.float32).pin_memory())
        self.chunks[c][k].copy_(loss, non_blocking=True)
        self.n += 1

    def extend(self, vals: torch.Tensor):
        """Append a 1-D device tensor of per-step losses (the graph step's device ring), stream-ordered, no host sync."""
        k0 = 0
        while k0 < vals.numel():
            c, k = divmod(self.n, self.CHUNK)
            if c == len(self.chunks):
                self.chunks.append(torch.empty(self.CHUNK, dtype=torch.float32).pin_memory())
            m = min(self.CHUNK - k, vals.numel() - k0)
            self.chunks[c][k:k + m].copy_(vals[k0:k0 + m], non_blocking=True)
            self.n += m
            k0 += m

    def values(self) -> torch.Tensor:
        if self.n == 0:
            return torch.empty(0)
        return torch.cat(self.chunks)[:self.n].clone()


_TRACE = _LossTrace()


_ENQUEUE = {"seconds": 0.0, "batches": 0, "graph_steps": 0}


def last_enqueue_ms_per_step() -> float:
    """Host time the most recent `train_one_epoch` call spent ENQUEUING one micro-batch (loop body only, before the one
    synchronising read of the loss sum at the end): the number that must stay below the GPU time of a step."""
    return 1e3 * _ENQUEUE["seconds"] / max(1, _ENQUEUE["batches"])


def last_graph_steps() -> int:
    """How many micro-batches of the most recent `train_one_epoch` call ran as one CUDA-graph replay each."""
    return int(_ENQUEUE.get("graph_steps", 0))


def last_step_losses() -> torch.Tensor:
    """Losses of every micro-batch of the most recent `train_one_epoch` call (fp32, CPU)."""
    return _TRACE.values()


class FusedStep:
    """Owns the flat Adam moments / step counter and runs the fused optimiser-side pass."""

    def __init__(self, model, optimizer, arena):
        self.model, self.opt, self.arena = model, optimizer, arena
        self.stats = torch.zeros(4, dtype=torch.float32, device=arena.flat.device)
        self.fusable = self._fusable()
        if self.fusable:
            self._adopt_state()

    def _fusable(self) -> bool:
        opt = self.opt
        if type(opt) not in (torch.optim.AdamW, torch.optim.Adam) or len(opt.param_groups) != 1:
            return False
        g = opt.param_groups[0]
        if g.get("amsgrad") or g.get("maximize") or g.get("differentiable"):
            return False
        ps = g["params"]
        return len(ps) == len(self.arena.params) and all(a is b for a, b in zip(ps, self.arena.params))

    def _adopt_state(self):
        ar, opt = self.arena, self.opt
        self.m = torch.zeros_like(ar.flat)
        self.v = torch.zeros_like(ar.flat)
        self.step = torch.zeros(1, dtype=torch.float32, device=ar.flat.device)
        mv, vv = ar.views(self.m), ar.views(self.v)
        with torch.no_grad():
            for p, a, b in zip(ar.params, mv, vv):
                st = opt.state.get(p)
                if st:                                    # resume: adopt existing moments
                    a.copy_(st["exp_avg"])
                    b.copy_(st["exp_avg_sq"])
                    self.step.fill_(float(st["step"]))
                opt.state[p] = {"step": self.step[0], "exp_avg": a, "exp_avg_sq": b}

    def still_valid(self, model, optimizer, arena) -> bool:
        if not (model is self.model and optimizer is self.opt and arena is self.arena and arena.valid()):
            return False
        if self.fusable:                                  # optimizer.load_state_dict() replaces the state tensors
            st = optimizer.state.get(arena.params[-1])
            if not st or st["exp_avg"].data_ptr() != self.m.data_ptr() + 4 * arena.offsets[-1]:
                return False
        return True

    def run(self, scaler, use_scaler: bool, grad_clip, ema):
        ar = self.arena
        dev = ar.flat.device
        st = _stream(dev)
        scale_ptr = scaler._scale.data_ptr() if use_scaler else None
        _lib.call("ddpm_param_reduce", ar.grad.data_ptr(), ar.numel, self.stats.data_ptr(), st)
        max_norm = float(grad_clip) if grad_clip is not None else 0.0
        ema_flat = None
        if ema is not None and isinstance(ema, EMA) and (ema._flat_ok(self.model) or ema._reflatten(self.model)):
            ema_flat = ema._flat
        if self.fusable:
            g = self.opt.param_groups[0]
            h = _lib.AdamHyper(float(g["lr"]), float(g["betas"][0]), float(g["betas"][1]), float(g["eps"]),
                               float(g["weight_decay"]), max_norm, float(ema.decay) if ema_flat is not None else 0.0,
                               1 if type(self.opt) is torch.optim.AdamW else 0)
            _lib.call("ddpm_param_update", ar.flat.data_ptr(), ar.grad.data_ptr(), self.m.data_ptr(), self.v.data_ptr(),
                      ema_flat.data_ptr() if ema_flat is not None else None, ar.numel, self.stats.data_ptr(),
                      self.step.data_ptr(), scale_ptr, C.byref(h), st)
            if ema is not None and ema_flat is None:
                ema.update(self.model)
        else:
            # any other optimiser: unscale+clip in one kernel, torch's own step, then the EMA kernel
            _lib.call("ddpm_grad_unscale_clip", ar.grad.data_ptr(), ar.numel, self.stats.data_ptr(), scale_ptr, max_norm, st)
            if float(self.stats[1].item()) == 0.0:
                self.opt.step()
            if ema is not None:
                ema.update(self.model)
        if use_scaler:
            # (the kernel also records stats[2] = the scale THIS step's gradients carried, for grad_norm())
            _lib.call("ddpm_scaler_update", scaler._scale.data_ptr(), scaler._growth_tracker.data_ptr(),
                      self.stats.data_ptr(), float(scaler.get_growth_factor()), float(scaler.get_backoff_factor()),
                      int(scaler.get_growth_interval()), st)
        GLOBAL_WCACHE.repack_all(st)      # packed weight copies are stale now: one batched launch refreshes them all
        ar.grad.zero_()                   # == optimizer.zero_grad(); grads stay attached (views)

    def grad_norm(self, scaler, use_scaler: bool) -> float:
        """||g||_2 of the unscaled gradients from the last reduction (diagnostic; one host sync)."""
        st = self.stats.tolist()                       # [sum g^2, found_inf, scale used by this step, -]
        s = st[2] if (use_scaler and st[2] > 0.0) else 1.0
        return st[0] ** 0.5 / s


def _get_fused(model, optimizer, arena) -> FusedStep:
    fs = getattr(model, "_ddpm_fused_step", None)
    if fs is None or not fs.still_valid(model, optimizer, arena):
        fs = FusedStep(model, optimizer, arena)
        object.__setattr__(model, "_ddpm_fused_step", fs)
    return fs


_COPY_STREAMS = {}
_STAGE_SLOTS = 3


def _staged_batches(dataloader, dev, max_batches):
    """Yields the loader's (x, y) pairs with the host->device copy of batch i+1 already in flight on a copy stream while
    step i computes: `x.to(dev, non_blocking=True)` on the compute stream (train_one_epoch.py:63 of the reference) puts
    0.25 ms of PCIe time per 6 MB batch in front of every step.  Only pinned CPU tensors are staged ahead (a pageable
    source blocks the host either way); nothing beyond `max_batches` is drawn from the loader.  The device side is a ring
    of three persistent buffers per batch shape (no allocator traffic, no record_stream): slot k is overwritten only after
    the compute stream has passed the step that read it."""
    key = str(dev)
    st = _COPY_STREAMS.get(key)
    if st is None:
        st = _COPY_STREAMS[key] = {"stream": torch.cuda.Stream(dev), "ring": {}}
    cs, rings = st["stream"], st["ring"]
    it = iter(dataloader)

    def stage(i):
        if (max_batches is not None) and (i >= max_batches):
            return None
        try:
            x, y = next(it)
        except StopIteration:
            return None
        if isinstance(x, torch.Tensor) and x.device.type == "cpu" and x.is_pinned():
            rk = (tuple(x.shape), x.dtype)
            ring = rings.get(rk)
            if ring is None:
                if len(rings) > 4:
                    rings.clear()
                ring = rings[rk] = {"buf": [torch.empty(x.shape, dtype=x.dtype, device=dev) for _ in range(_STAGE_SLOTS)],
                                    "free": [None] * _STAGE_SLOTS, "n": 0}
            k = ring["n"] % _STAGE_SLOTS
            ring["n"] += 1
            if ring["free"][k] is not None:
                cs.wait_event(ring["free"][k])            # the step that read this slot has been passed by the compute stream
            with torch.cuda.stream(cs):
                ring["buf"][k].copy_(x, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(cs)
            return ring["buf"][k], y, ev, (ring, k)
        return x, y, None, None

    i = 0
    nxt = stage(0)
    while nxt is not None:
        x, y, ev, slot = nxt
        nxt = stage(i + 1)
        if ev is not None:
            torch.cuda.current_stream(dev).wait_event(ev)
        yield x, y
        if slot is not None:                                  # everything that reads x has been enqueued by now
            done = torch.cuda.Event()
            done.record(torch.cuda.current_stream(dev))
            slot[0]["free"][slot[1]] = done
        i += 1


# ------------------------------------------------------------------------------------------------------------------
# The whole optimiser step as ONE CUDA graph (SURVEY.md section 7 step 9; reference loop body train_one_epoch.py:61-121).
# Eager, a step is ~300 kernel launches enqueued by ~6.4 ms of host work with ~240 inter-kernel gaps of ~2 us; captured
# (timestep draw, q_sample, UNet forward + backward incl. the side-stream weight gradients, the fused unscale / clip /
# AdamW / EMA / scaler pass, the weight repack and the gradient zeroing) it replays with 0.02 ms of host work:
# 12.00 -> 11.66 ms per step at B = 128 (tools/train_graph_probe.py).  Everything the step mutates lives at fixed device
# addresses (parameter / gradient / moment / EMA arenas, scaler scale, dropout RNG state, pooled activations); the batch
# is copied into a static input buffer, the loss goes to a device ring that is drained without a host sync, torch's CUDA
# generator is graph-safe (`randint` / `randn_like` advance their Philox offset per replay).
# Used when the step is a pure function of device state: single process, no gradient accumulation, constant
# hyper-parameters, fused optimiser, no overrides or hooks on the model / diffusion objects; a configuration runs eagerly
# until an epoch call has ended with at least two steps of it behind (lazy initialisation, pools), then it is captured.  Any change of configuration re-captures; DDPM_B200_TRAIN_GRAPH=0 turns it off.
# ------------------------------------------------------------------------------------------------------------------
class _GraphStep:
    RING = 1024

    def __init__(self, key, x: torch.Tensor):
        dev = x.device
        self.key = key
        self.x = torch.empty_like(x, memory_format=torch.contiguous_format)
        self.loss_sum = torch.zeros((), dtype=torch.float32, device=dev)
        self.step_loss = torch.zeros((), dtype=torch.float32, device=dev)
        self.ring = torch.zeros(self.RING, dtype=torch.float32, device=dev)
        self.idx = torch.zeros(1, dtype=torch.int64, device=dev)
        self.pending = 0                                  # ring entries not yet handed to the loss trace
        self.pos = 0                                      # host mirror of the device-side ring position
        self.graph = None

    def capture(self, body):
        def whole():
            loss = body(self.x)
            self.step_loss.copy_(loss)
            self.loss_sum.add_(self.step_loss)
            self.ring.index_copy_(0, self.idx, self.step_loss.reshape(1))
            self.idx.add_(1).remainder_(self.RING)
        g = torch.cuda.CUDAGraph()
        n0 = _lib.launch_count(reset=False)
        # The graph bakes the ADDRESSES of the pooled activation buffers it was captured with.  Record them and take them out of
        # the shared pool afterwards: eager work (a forward whose activations are still saved for a backward, a sampler) must
        # never be handed a buffer that a replay overwrites.
        used, orig_get = [], POOL.get

        def _recording_get(key, device):
            t = orig_get(key, device)
            used.append((key, t))
            return t
        POOL.get = _recording_get
        try:
            with torch.cuda.graph(g, capture_error_mode="global"):
                whole()
        finally:
            del POOL.get                                  # back to the class method
        self.n_launch = _lib.launch_count(reset=False) - n0    # library kernels inside the graph (credited per replay)
        import gc
        gc.collect()                                      # activation views caught in reference cycles go back to the pool now
        self.owned, seen = [], set()
        for key, t in used:
            if t.data_ptr() in seen:
                continue
            seen.add(t.data_ptr())
            lst = POOL.free.get(key)
            if lst:
                for k, u in enumerate(lst):
                    if u is t:
                        lst.pop(k)
                        break
            self.owned.append(t)
        self.graph = g

    def run(self, x: torch.Tensor):
        self.x.copy_(x, non_blocking=True)
        self.graph.replay()
        _lib.lib.ddpm_launch_count_add(self.n_launch)
        self.pos = (self.pos + 1) % self.RING
        self.pending += 1
        if self.pending == self.RING:
            self.drain()

    def drain(self):
        """Hand the ring entries [pos - pending, pos) (modulo RING, oldest first) to the loss trace; stream-ordered."""
        if self.pending:
            lo = (self.pos - self.pending) % self.RING
            if lo < self.pos:
                _TRACE.extend(self.ring[lo:self.pos])
            else:
                _TRACE.extend(self.ring[lo:])
                if self.pos:
                    _TRACE.extend(self.ring[:self.pos])
            self.pending = 0


def _graph_enabled() -> bool:
    return os.environ.get("DDPM_B200_TRAIN_GRAPH", "1") != "0"


def _pure_step(model, diffusion) -> bool:
    """A captured step replays device work only: it is valid when `diffusion.sample_timesteps`, `diffusion.loss_simple` and
    `model.forward` are this package's own methods (which draw from torch's CUDA generator and launch kernels) -- not
    instance-level overrides or hooks, whose host-side effects (a Python iterator feeding noise, logging, ...) a replay
    would silently skip."""
    from ..model.difussion_class import Diffusion
    from ..model.unet_backbone import UNetDenoiser
    if type(diffusion) is not Diffusion or type(model) is not UNetDenoiser:
        return False
    if any(k in vars(diffusion) for k in ("sample_timesteps", "loss_simple", "q_sample")) or "forward" in vars(model):
        return False
    for m in model.modules():
        if m._forward_hooks or m._forward_pre_hooks or m._backward_hooks or getattr(m, "_backward_pre_hooks", None):
            return False
    return True


def _header(probe_timesteps):
    print("┆   {:>8} | {:>9} | {:>8} | {:>8} | {:>10}{}".format(
        "step", "lr", "loss", "dt(ms)", "grad_norm", (" | probes[t]" if probe_timesteps else "")))
    print("┆   " + "─" * 72)


def train_one_epoch(model, diffusion, dataloader, optimizer, *, scaler=None, ema=None, device: str = "cuda",
                    max_batches: int | None = None, grad_clip: float | None = 1.0, use_autocast: bool = True,
                    grad_accum_steps: int = 1, use_channels_last: bool = False, on_oom: str = "skip",
                    base_lr: float | None = None, warmup_steps: int | None = None, global_step: int = 0,
                    log_every: int = 0, probe_timesteps: list[int] | None = None, log_mem: bool = False,
                    log_grad_norm: bool = False):
    """train_one_epoch.py:11-168.  Returns (avg_loss, n_batches, n_images, global_step)."""
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("ddpm_b200.train_one_epoch is CUDA-only (sm_100a); there is no CPU fallback")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    model.train()
    # use_channels_last only affects the *input* layout here: kernels are NHWC internally and the
    # parameters must stay contiguous OIHW views of the flat arena.
    rank, world = _dist.world()
    verbose = rank == 0
    grad_accum_steps = max(1, int(grad_accum_steps))
    arena = ensure_arena(model)
    if arena is None:
        raise RuntimeError("ddpm_b200.train_one_epoch needs an fp32 CUDA model with all parameters trainable")
    fused = _get_fused(model, optimizer, arena)
    arena.attach_grads(zero=True)                      # == optimizer.zero_grad(set_to_none=True)
    sync = _dist.attach_grad_sync(model, arena) if world > 1 else None
    use_scaler = bool(use_autocast and (scaler is not None))

    loss_sum = torch.zeros((), dtype=torch.float32, device=dev)
    _TRACE.reset()
    # one-graph-per-step path (see _GraphStep): only when a step is a pure function of device state, and only in a single
    # process -- capturing the bucketed NCCL all-reduces with the step hung on 2 GPUs (DESIGN §6.3), so multi-process runs
    # stay eager
    graph_ok = (_graph_enabled() and world == 1 and grad_accum_steps == 1 and fused.fusable and on_oom == "skip"
                and not ((base_lr is not None) and (warmup_steps is not None) and (warmup_steps > 0) and global_step < warmup_steps)
                and not getattr(model, "_ddpm_train_graph_failed", False) and _pure_step(model, diffusion))
    gcache = getattr(model, "_ddpm_train_graphs", None)   # key -> {"key", "warm", "gs"}; a few configurations stay captured
    if gcache is None:
        gcache = {}
        object.__setattr__(model, "_ddpm_train_graphs", gcache)
    gstate = None
    if any(v.get("gs") is not None for v in gcache.values()):
        GLOBAL_WCACHE.repack_all(_stream(dev))            # parameters may have been changed in place between epochs
    n_graph_steps = 0
    last_x = None
    n_seen_batches, n_seen_images = 0, 0
    did_header = False
    if log_every and global_step == 0:
        with torch.no_grad():
            xb = torch.randn(32, 3, diffusion.img_size, diffusion.img_size, device=dev)
            base = float((xb ** 2).mean().item())
        if verbose:
            print("┆ In-epoch statistics")
            print("┆   (baseline)  ε-MSE ≈ {:.3f}  (esperado ~1.0)".format(base))
            _header(probe_timesteps)
        did_header = True

    t_loop = time.perf_counter()
    for i, (x, _) in enumerate(_staged_batches(dataloader, dev, max_batches)):
        if (max_batches is not None) and (i >= max_batches):
            break
        try:
            t_start = time.perf_counter()
            x = x.to(dev, non_blocking=True)
            if use_channels_last:
                x = x.to(memory_format=torch.channels_last)
            B = x.size(0)
            step_now = ((i + 1) % grad_accum_steps) == 0
            if not arena.grads_attached():
                arena.attach_grads(zero=True)
            if sync is not None:
                if step_now:
                    sync.begin()
                else:
                    sync.reset()

            gs = None
            if graph_ok:
                g0 = optimizer.param_groups[0]
                gkey = (GRAPH_EPOCH[0], id(model), id(diffusion), id(optimizer), id(scaler) if use_scaler else None, id(ema), id(fused),
                        tuple(x.shape), x.dtype, x.is_contiguous(), bool(use_autocast), use_scaler, grad_clip,
                        float(g0["lr"]), tuple(g0["betas"]), float(g0["eps"]), float(g0["weight_decay"]),
                        float(getattr(ema, "decay", 0.0)) if ema is not None else None,
                        (scaler.get_growth_factor(), scaler.get_backoff_factor(), scaler.get_growth_interval()) if use_scaler else None,
                        # every buffer the graph reads or writes must still be where it was at capture
                        arena.flat.data_ptr(), arena.grad.data_ptr(), fused.m.data_ptr(), fused.step.data_ptr(),
                        scaler._scale.data_ptr() if (use_scaler and scaler._scale is not None) else None,
                        ema._flat.data_ptr() if (ema is not None and getattr(ema, "_flat", None) is not None) else None)
                if gstate is None or gstate["key"] != gkey:
                    if gstate is not None and gstate.get("gs") is not None:
                        gstate["gs"].drain()
                        loss_sum += gstate["gs"].loss_sum
                    gstate = gcache.get(gkey)
                    if gstate is None:
                        while len(gcache) >= 4:               # oldest configuration goes (its graph and private pool with it)
                            gcache.pop(next(iter(gcache)))
                        gstate = gcache[gkey] = {"key": gkey, "warm": 0, "gs": None}
                    if gstate["gs"] is not None:
                        gstate["gs"].loss_sum.zero_()
                gs = gstate["gs"]
                last_x = x
            if gs is not None:
                gs.run(x)
                gstate["replays"] = gstate.get("replays", 0) + 1
                n_graph_steps += 1
                loss = gs.step_loss
            else:
                if gstate is not None and graph_ok:
                    gstate["warm"] += 1
                t = diffusion.sample_timesteps(B, device=dev)
                with autocast_ctx(device="cuda", enabled=bool(use_autocast), dtype="bf16"):
                    loss = diffusion.loss_simple(model, x, t) / grad_accum_steps
                if use_scaler:
                    scaler.scale(loss).backward()
                else:
                    loss.backward()

            gnorm = None
            if gs is not None:
                if log_grad_norm:
                    gnorm = fused.grad_norm(scaler, use_scaler)
                global_step += 1
            elif step_now:
                if (base_lr is not None) and (warmup_steps is not None) and (warmup_steps > 0):
                    lr = base_lr * min(1.0, (global_step + 1) / warmup_steps)
                    for g in optimizer.param_groups:
                        g["lr"] = lr
                if sync is not None:
                    sync.finish()
                fused.run(scaler if use_scaler else None, use_scaler, grad_clip, ema)
                if log_grad_norm:
                    gnorm = fused.grad_norm(scaler, use_scaler)
                global_step += 1

            if gs is None:
                step_loss = loss.detach().float() * grad_accum_steps
                loss_sum += step_loss
                _TRACE.push(step_loss)
            n_seen_batches += 1
            n_seen_images += B

            if log_every and (global_step % log_every == 0) and step_now:
                if not did_header:
                    if verbose:
                        print("┆ In-epoch statistics")
                        _header(probe_timesteps)
                    did_header = True
                probe_msg = ""
                if probe_timesteps:
                    with torch.no_grad(), autocast_ctx(device="cuda", enabled=True, dtype="bf16"):
                        probes = []
                        for tau in probe_timesteps:
                            t_fix = torch.full((B,), int(tau), device=dev, dtype=torch.long)
                            probes.append(diffusion.loss_simple(model, x, t_fix).detach().float())
                        # ONE host read for all probes (the reference syncs once per probe, train_one_epoch.py:134-142)
                        vals = [f"t={tau}:{v:.3f}" for tau, v in zip(probe_timesteps, torch.stack(probes).tolist())]
                        probe_msg = " | " + " ".join(vals)
                mem_msg = ""
                if log_mem:
                    alloc, reserv = gpu_mem_mb("cuda")
                    mem_msg = f" | mem={alloc:.0f}/{reserv:.0f}MB"
                lr_now = optimizer.param_groups[0]["lr"]
                dt = (time.perf_counter() - t_start) * 1000.0
                gn_str = (f"{gnorm:.2e}" if (gnorm is not None) else "—")
                loss_val = (loss.detach() * grad_accum_steps).item()
                if verbose:
                    print("┆   {:8d} | {:9.2e} | {:8.4f} | {:8.1f} | {:>10}{}{}".format(
                        global_step, lr_now, loss_val, dt, gn_str, mem_msg, probe_msg))
        except RuntimeError as e:
            if ("CUDA out of memory" in str(e)) and (on_oom == "skip"):
                import gc
                gc.collect()
                torch.cuda.empty_cache()
                if verbose:
                    print(f"[WARN][OOM] Batch {i} omitido. Limpié cache y sigo…")
                if arena.grad is not None:
                    arena.grad.zero_()
                continue
            raise

    _ENQUEUE["seconds"], _ENQUEUE["batches"] = time.perf_counter() - t_loop, n_seen_batches
    _ENQUEUE["graph_steps"] = n_graph_steps
    if gstate is not None and gstate.get("gs") is not None:
        gstate["gs"].drain()
        loss_sum += gstate["gs"].loss_sum
    avg_loss = float(loss_sum.item()) / max(1, n_seen_batches)
    # Capture for the NEXT call, at a quiet point: the loop is over, the loss read above has synchronised, nothing of the last
    # iteration is alive.  (Capturing in the middle of the loop was refused by the runtime -- "operation failed due to a previous
    # error during capture" in every capture-error mode -- while the identical body captured right after an epoch call; the
    # cost of a capture, ~40 ms, also belongs outside the steps.)
    if graph_ok and gstate is not None and gstate.get("gs") is None and gstate["warm"] >= 2 and last_x is not None:
        xs0, Bc = last_x, last_x.size(0)
        x = loss = None                                   # noqa: F841  (drop the last iteration's tensors)

        def _body(xs):
            tt = diffusion.sample_timesteps(Bc, device=dev)
            with autocast_ctx(device="cuda", enabled=bool(use_autocast), dtype="bf16"):
                ls = diffusion.loss_simple(model, xs, tt)
            if use_scaler:
                scaler.scale(ls).backward()
            else:
                ls.backward()
            fused.run(scaler if use_scaler else None, use_scaler, grad_clip, ema)
            return ls.detach().float()
        try:
            # A configuration that changes every epoch (a per-epoch lr schedule bakes a new lr into the key) would be captured
            # again and again without ever being replayed, each capture holding its own activation buffers: after two captured
            # graphs that were never replayed the model stays eager; at most two captured configurations are kept.
            captured = [v for v in gcache.values() if v.get("gs") is not None]
            if sum(1 for v in captured if v.get("replays", 0) == 0) >= 2:
                for v in captured:
                    if v.get("replays", 0) == 0:
                        v["gs"] = None
                raise RuntimeError("the step's configuration changes from call to call (captured graphs were never replayed)")
            for v in captured[:max(0, len(captured) - 1)]:
                v["gs"] = None
            arena.attach_grads(zero=True)
            cand = _GraphStep(gstate["key"], xs0)
            cand.capture(_body)
            gstate["gs"] = cand
            gstate["replays"] = 0
        except Exception as ex:                           # an op that cannot be captured: stay eager from now on
            object.__setattr__(model, "_ddpm_train_graph_failed", True)
            if verbose:
                print(f"[ddpm_b200] CUDA-graph capture of the train step failed ({type(ex).__name__}: "
                      f"{str(ex).splitlines()[0]}); running eagerly")
            if arena.grad is not None:
                arena.grad.zero_()
    return avg_loss, n_seen_batches, n_seen_images, global_step
