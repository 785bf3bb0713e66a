"""Data-parallel plumbing (one process per GPU, torch.distributed / NCCL over NVLink).

The reference is single-GPU (SURVEY.md §2.1); the path shards naturally:
  * training: pure data parallelism.  Each rank runs fwd/bwd on its own images; the only exchange
    step is the all-reduce (average) of the flat fp32 gradient arena, issued bucket by bucket on a
    side stream while the rest of backward is still running, then the (redundant, identical)
    fused unscale+clip+AdamW+EMA pass runs on every rank -- found-inf and the clipping norm are
    computed on the reduced gradients, so all ranks take the same decision with no extra collective;
  * sampling: batch-sharded, no communication (`shard_range`).
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import torch
import torch.distributed as dist


def world() -> Tuple[int, int]:
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_range(n: int, rank: Optional[int] = None, world_size: Optional[int] = None) -> Tuple[int, int]:
    """Rows [lo, hi) of an n-image batch owned by `rank` (contiguous, sizes differ by at most 1)."""
    r, w = world()
    rank = r if rank is None else rank
    world_size = w if world_size is None else world_size
    base, rem = divmod(n, world_size)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def make_buckets(numel: int, bucket_elems: int, tail_elems: int = 0, tail_bucket_elems: int = 0) -> List[Tuple[int, int]]:
    """[start, end) element ranges covering the arena from its END to its START (backward order).

    The gradients at the START of the arena (in_conv, time_mlp, the first encoder level) become final last, so whatever
    bucket holds them cannot be hidden behind backward: its all-reduce is the exposed tail in front of the optimiser
    pass.  With `tail_elems` > 0 the first `tail_elems` elements are therefore cut into small buckets of
    `tail_bucket_elems` -- the reduction of all but the last small piece still overlaps the end of backward, and the
    exposed piece is a few hundred KB instead of a full bucket."""
    out, end = [], numel
    tail_elems = min(max(0, tail_elems), numel)
    while end > tail_elems:
        start = max(tail_elems, end - bucket_elems)
        out.append((start, end))
        end = start
    step = max(1, tail_bucket_elems or bucket_elems)
    while end > 0:
        start = max(0, end - step)
        out.append((start, end))
        end = start
    return out


class GradSync:
    """Bucketed gradient averaging over a flat arena, overlapped with backward.

    `module_spans` maps id(module) -> (lo, hi) element span of that module's parameters; modules
    report completion through `progress(module)` (engine.unet_backward) and a bucket is reduced as
    soon as every span that intersects it is final.  `progress(None)` / `finish()` flush the rest."""

    def __init__(self, flat_grad: torch.Tensor, module_spans: dict, bucket_bytes: int = 16 << 20, group=None,
                 tail_bytes: int = 4 << 20, tail_bucket_bytes: int = 4 << 20):
        self.g = flat_grad
        self.group = group
        self.spans = module_spans
        # Measured on 8 B200 (profiles/r2_timeline_dp8*.txt): with plain 16 MB buckets the third bucket cannot start before
        # the first encoder level is done, i.e. at the very end of backward -- 181 us of exposed all-reduce.  Cutting the
        # first 12 MB into 2 MB buckets halves the exposed wait (100 us) but the nine NCCL kernels steal more SM time from
        # the overlapped backward than that saves (12.59 vs 12.50 ms per step).  One boundary at 4 MB keeps four launches:
        # [4 MB, ...) goes out while the first encoder level's backward (~1 ms) is still running, only [0, 4 MB)
        # (time MLP, in/out convolutions, first encoder level) is exposed.
        self.buckets = make_buckets(flat_grad.numel(), max(1, bucket_bytes // 4), tail_bytes // 4, max(1, tail_bucket_bytes // 4))
        self.cuda = flat_grad.is_cuda
        self.comm = torch.cuda.Stream(flat_grad.device) if self.cuda else None
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.reset()

    def reset(self):
        self.done_ids = set()
        self.next = 0
        self.handles = []
        self.active = False

    def begin(self):
        self.reset()
        self.active = True

    def _final_low(self) -> int:
        """Lowest offset such that every reported span at or above it is complete."""
        low = self.g.numel()
        for mid, (lo, hi) in sorted(self.spans.items(), key=lambda kv: -kv[1][0]):
            if mid in self.done_ids:
                low = lo
            else:
                break
        return low

    def _launch(self, start: int, end: int):
        view = self.g[start:end]
        if self.world == 1:
            return
        if self.cuda:
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(self.g.device))
            self.comm.wait_event(ev)
            with torch.cuda.stream(self.comm):
                dist.all_reduce(view, op=dist.ReduceOp.AVG, group=self.group)
        else:
            dist.all_reduce(view, op=dist.ReduceOp.SUM, group=self.group)
            view.mul_(1.0 / self.world)

    def progress(self, module):
        if not self.active:
            return
        if module is None:
            self.finish()
            return
        self.done_ids.add(id(module))
        low = self._final_low()
        while self.next < len(self.buckets) and self.buckets[self.next][0] >= low:
            self._launch(*self.buckets[self.next])
            self.next += 1

    def finish(self):
        if not self.active:
            return
        while self.next < len(self.buckets):
            self._launch(*self.buckets[self.next])
            self.next += 1
        if self.cuda and self.world > 1:
            torch.cuda.current_stream(self.g.device).wait_stream(self.comm)
        self.active = False


def module_spans(model: torch.nn.Module, arena) -> dict:
    """Parameter spans of the sub-modules that `engine.unet_backward` reports as they complete."""
    from . import engine
    spans = {}

    def span_of(params):
        offs = [(arena.offset_of[id(p)], arena.offset_of[id(p)] + p.numel()) for p in params if id(p) in arena.offset_of]
        return (min(o[0] for o in offs), max(o[1] for o in offs)) if offs else None

    mods = []
    if hasattr(model, "downs") and hasattr(model, "ups"):
        for lvl in list(model.downs) + list(model.ups):
            mods += list(lvl.blocks)
            for name in ("down", "up"):
                m = getattr(lvl, name, None)
                if m is not None and not isinstance(m, torch.nn.Identity):
                    mods.append(m)
        mods += [m for m in model.mid if not isinstance(m, torch.nn.Identity)]
    for m in mods:
        s = span_of(list(m.parameters()))
        if s is not None:
            spans[id(m)] = s
    return spans


def attach_grad_sync(model: torch.nn.Module, arena, bucket_bytes: int = 16 << 20, group=None) -> Optional[GradSync]:
    """Create (once) the GradSync of `model`; returns None when not running distributed."""
    _, w = world()
    if w == 1:
        return None
    gs = getattr(model, "_ddpm_grad_sync", None)
    if gs is None or gs.g.data_ptr() != arena.grad.data_ptr():
        gs = GradSync(arena.grad, module_spans(model, arena), bucket_bytes, group)
        object.__setattr__(model, "_ddpm_grad_sync", gs)
        object.__setattr__(model, "_ddpm_grad_progress", gs.progress)
    return gs
