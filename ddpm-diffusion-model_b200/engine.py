"""Host-side executor of the UNet hot path on the C ABI (libddpm_b200.so).

Data layout in HBM
  * activations: NHWC, element type bf16 (autocast) or fp32, every buffer carries a one-pixel zero
    halo (`[N][H+2][W+2][pitch]`) that no kernel ever writes -> 3x3 convolutions need no bounds
    logic on the tensor-core path and skip-concatenation is a channel slice of one wide buffer
    (producers write at a channel offset; `torch.cat` of unet_backbone.py:206 disappears);
  * parameters / gradients: fp32 in the reference's OIHW layout (state_dict compatible); packed
    copies `[Cout][tap][Cin]` (fprop) and `[Cin][tap'][Cout]` (dgrad) in the activation dtype are
    cached per parameter version;
  * the time path (sinusoid -> MLP -> per-block time_proj) is fp32 `[B][C]`.

The forward functions return `(out, saved)`; the hand-derived backward functions consume `saved`
in reverse order.  Nothing here touches the oracle and nothing falls back to ATen math.
"""
from __future__ import annotations

import ctypes as C
import weakref
from typing import Dict, List, Optional, Tuple

import torch

from . import _lib
from ._lib import Tensor as CT

_TORCH = {_lib.F32: torch.float32, _lib.BF16: torch.bfloat16}
_ESZ = {_lib.F32: 4, _lib.BF16: 2}


# ----------------------------------------------------------------------------------------------
# buffers
# ----------------------------------------------------------------------------------------------
class _Pool:
    """Recycles halo-zeroed activation buffers per (device, dtype, shape).  A buffer's interior is
    always fully overwritten by its producer and its halo is never written, so no memset is needed
    after the first allocation."""

    def __init__(self):
        self.free: Dict[tuple, List[torch.Tensor]] = {}
        self.enabled = True
        self.misses = 0           # allocations (each costs a cudaMalloc-cache lookup + a zero-fill kernel)

    def get(self, key, device):
        lst = self.free.get(key)
        if lst:
            return lst.pop()
        _, dt, shape = key
        self.misses += 1
        return torch.zeros(shape, dtype=dt, device=device)

    def put(self, key, t):
        if self.enabled:
            self.free.setdefault(key, []).append(t)

    def clear(self):
        self.free.clear()
        GRAPH_EPOCH[0] += 1       # captured CUDA graphs hold raw addresses of pooled buffers: never replay them after this


# Bumped whenever memory that a captured train-step graph may reference by address is released (pool cleared, split-K
# workspace re-allocated); `train_one_epoch` keys its graphs on it.
GRAPH_EPOCH = [0]
POOL = _Pool()


class _Buf:
    __slots__ = ("t", "key")

    def __init__(self, t, key):
        self.t, self.key = t, key

    def __del__(self):
        if self.key is None:          # wrapped (non-pooled) tensor
            return
        try:
            POOL.put(self.key, self.t)
        except Exception:
            pass


class Act:
    """An NHWC view (possibly a channel slice) of a pooled buffer."""
    __slots__ = ("buf", "N", "H", "W", "C", "pitch", "c0", "halo", "dt", "_d")

    def __init__(self, buf, N, H, W, C, pitch, c0, halo, dt):
        self.buf, self.N, self.H, self.W, self.C = buf, N, H, W, C
        self.pitch, self.c0, self.halo, self.dt = pitch, c0, halo, dt
        self._d = None

    @staticmethod
    def new(N, H, W, C, dt, device, halo=1) -> "Act":
        shape = (N, H + 2 * halo, W + 2 * halo, C)
        key = (str(device), _TORCH[dt], shape)
        return Act(_Buf(POOL.get(key, device), key), N, H, W, C, C, 0, halo, dt)

    @staticmethod
    def wrap(t: torch.Tensor, N, H, W, C, dt, halo=0) -> "Act":
        """View an existing contiguous tensor [N,H,W,C] (no pooling)."""
        b = _Buf.__new__(_Buf)
        b.t, b.key = t, None
        a = Act(b, N, H, W, C, C, 0, halo, dt)
        return a

    def slice(self, c0, C) -> "Act":
        return Act(self.buf, self.N, self.H, self.W, C, self.pitch, self.c0 + c0, self.halo, self.dt)

    @property
    def ptr(self) -> int:
        return self.buf.t.data_ptr() + self.c0 * _ESZ[self.dt]

    def desc(self) -> CT:
        if self._d is None:
            self._d = CT(self.ptr, self.N, self.H, self.W, self.C, self.pitch, self.halo)
        return self._d

    def interior(self) -> torch.Tensor:
        """torch view [N,H,W,C] (debug / tests)."""
        h = self.halo
        t = self.buf.t
        return t[:, h:t.shape[1] - h, h:t.shape[2] - h, self.c0:self.c0 + self.C]


def _null_tensor() -> CT:
    return CT(None, 0, 0, 0, 0, 0, 0)


_NULL = _null_tensor()


# ----------------------------------------------------------------------------------------------
# per-call execution context
# ----------------------------------------------------------------------------------------------
class WeightCache:
    """Packed (fprop / dgrad) copies of conv and linear weights, keyed by parameter identity and
    refreshed when the parameter's version counter or the owner's epoch changes."""

    def __init__(self):
        self.entries: Dict[tuple, tuple] = {}
        self.up2x: Dict[tuple, tuple] = {}
        self.epoch = 0
        self._table = None            # (device uint8 tensor of ddpm_pack_entry[], n, signature)

    def bump(self):
        self.epoch += 1

    def repack_all(self, stream: int) -> bool:
        """After an in-place optimiser step every packed copy is stale at once: refresh all live entries with ONE
        launch (ddpm_pack_weights_batched) instead of one launch per weight on the next forward.  Returns False
        (and leaves the lazy per-weight path to do it) if nothing is cached yet."""
        self.epoch += 1
        live = [(k, e) for k, e in self.entries.items()
                if e[4]() is not None and e[3].data_ptr() == e[4]().data_ptr() and e[4]().is_cuda]
        if not live:
            return False
        sig = tuple((k, e[3].data_ptr(), e[1].data_ptr(), e[2].data_ptr() if e[2] is not None else 0) for k, e in live)
        if self._table is None or self._table[2] != sig:
            arr = (_lib.PackEntry * len(live))()
            for i, (k, e) in enumerate(live):
                _, dt, cin_pad, cout_pad = k
                wd = e[3]
                co, ci = wd.shape[0], wd.shape[1]
                taps = wd.shape[2] * wd.shape[3] if wd.dim() == 4 else 1
                arr[i] = _lib.PackEntry(wd.data_ptr(), e[1].data_ptr(), e[2].data_ptr() if e[2] is not None else None,
                                        co, ci, taps, max(ci, cin_pad), max(co, cout_pad), dt)
            host = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8)
            self._table = (host.to(live[0][1][1].device), len(live), sig)
        _lib.call("ddpm_pack_weights_batched", self._table[0].data_ptr(), self._table[1], stream)
        for k, e in live:
            w = e[4]()
            self.entries[k] = ((w._version, self.epoch, w.data_ptr()), e[1], e[2], e[3], e[4])
        return True

    def get_up2x(self, E: "Exec", w: torch.Tensor, dt: int) -> torch.Tensor:
        """[4][Cout][4][Cin] phase weights of `conv3x3(nearest x2 (x))` evaluated on the low-resolution x
        (ddpm_pack_weights_up2x); refreshed lazily when the parameter's version or the cache epoch moves on."""
        key = (id(w), dt)
        ent = self.up2x.get(key)
        if ent is not None and ent[2]() is not w:
            ent = None
        stamp = (w._version, self.epoch, w.data_ptr())
        if ent is not None and ent[0] == stamp:
            return ent[1]
        co, ci = w.shape[0], w.shape[1]
        buf = ent[1] if ent is not None else torch.empty((4, co, 4, ci), dtype=_TORCH[dt], device=w.device)
        wd = w.detach()
        if not wd.is_contiguous():
            wd = wd.contiguous()
        _lib.call("ddpm_pack_weights_up2x", wd.data_ptr(), co, ci, buf.data_ptr(), dt, E.stream)
        if ent is None and len(self.up2x) > 32:
            for k in [k for k, e in self.up2x.items() if e[2]() is None]:
                del self.up2x[k]
        self.up2x[key] = (stamp, buf, weakref.ref(w))
        return buf

    def get(self, E: "Exec", w: torch.Tensor, dt: int, need_dgrad: bool, cin_pad: int = 0, cout_pad: int = 0):
        key = (id(w), dt, cin_pad, cout_pad)
        ent = self.entries.get(key)
        if ent is not None and ent[4]() is not w:          # id() reused by a new parameter object
            ent = None
        stamp = (w._version, self.epoch, w.data_ptr())
        if ent is not None and ent[0] == stamp and (ent[2] is not None or not need_dgrad):
            return ent[1], ent[2]
        if ent is None and len(self.entries) > 64:
            for k in [k for k, e in self.entries.items() if e[4]() is None]:
                del self.entries[k]
        co, ci = w.shape[0], w.shape[1]
        kh, kw = (w.shape[2], w.shape[3]) if w.dim() == 4 else (1, 1)
        tdt = _TORCH[dt]
        n_el = max(co, cout_pad) * max(ci, cin_pad) * kh * kw
        fwd = ent[1] if ent is not None and ent[1] is not None else torch.empty(n_el, dtype=tdt, device=w.device)
        dg = None
        if need_dgrad:
            dg = ent[2] if ent is not None and ent[2] is not None else torch.empty(n_el, dtype=tdt, device=w.device)
        wd = w.detach()
        if not wd.is_contiguous():
            wd = wd.contiguous()
        _lib.call("ddpm_pack_weights", wd.data_ptr(), co, ci, kh, kw, fwd.data_ptr(),
                  dg.data_ptr() if dg is not None else None, dt, cin_pad, cout_pad, E.stream)
        self.entries[key] = (stamp, fwd, dg, wd, weakref.ref(w))
        return fwd, dg


GLOBAL_WCACHE = WeightCache()
_WORKSPACES: Dict[str, torch.Tensor] = {}


class Exec:
    """Everything one forward(+backward) needs: dtype, stream, RNG state, weight cache, flags."""

    def __init__(self, device, dt: int, training: bool, need_grad: bool, wcache: Optional[WeightCache] = None,
                 rng: Optional[torch.Tensor] = None, prefer_tc: bool = True):
        self.device = device
        self.dt = dt
        self.tdt = _TORCH[dt]
        self.training = training
        self.need_grad = need_grad
        self.wcache = wcache if wcache is not None else GLOBAL_WCACHE
        self.rng = rng
        self.prefer_tc = 1 if prefer_tc else 0
        self.use_tc = bool(prefer_tc) and dt == _lib.BF16     # tcgen05 kernels (channel padding to 16)
        self.stream = _lib.stream_for(device)

    # ---- allocation helpers
    def act(self, N, H, W, C, halo=1) -> Act:
        return Act.new(N, H, W, C, self.dt, self.device, halo)

    def f32(self, *shape) -> torch.Tensor:
        return torch.empty(shape, dtype=torch.float32, device=self.device)

    def workspace(self, nbytes: int) -> torch.Tensor:
        """Scratch for split-K partials; one growing buffer per device (stream-ordered reuse)."""
        key = str(self.device)
        ws = _WORKSPACES.get(key)
        if ws is None or ws.numel() < nbytes:
            ws = torch.empty(max(nbytes, 32 << 20), dtype=torch.uint8, device=self.device)
            _WORKSPACES[key] = ws
            GRAPH_EPOCH[0] += 1
        return ws

    def vec(self, t: torch.Tensor, B: int, Cn: int) -> Act:
        """fp32 [B][C] tensor as an H=W=1 activation (time path)."""
        return Act.wrap(t, B, 1, 1, Cn, _lib.F32, 0)


_SIDE_STREAMS: Dict[str, "torch.cuda.Stream"] = {}


def fuse_skip_enabled() -> bool:
    import os
    return os.environ.get("DDPM_B200_FUSE_SKIP", "1") != "0"


def overlap_enabled() -> bool:
    import os
    return os.environ.get("DDPM_B200_WGRAD_OVERLAP", "1") != "0"


def _event_on(stream) -> "torch.cuda.Event":
    ev = torch.cuda.Event()
    ev.record(stream)
    return ev


def wgrad_async(E: "Exec", after: "torch.cuda.Event", fn) -> "torch.cuda.Event":
    """Run `fn` (weight-gradient launches) on the per-device side stream once `after` (a main-stream event) has
    completed; returns the side-stream event that marks their completion.  The weight gradients are off the
    critical path of backward (only the optimiser needs them), and the tensor-core wgrad kernel (TMA + MMA, one
    178 KB CTA per SM) leaves the ALU/LSU and two CTA slots per SM free -- exactly what the issue-bound
    GroupNorm backward running next on the main stream needs."""
    key = str(E.device)
    side = _SIDE_STREAMS.get(key)
    if side is None:
        # high priority: when a wgrad and a GroupNorm backward become runnable at the same moment the 178 KB wgrad
        # CTAs must be placed first -- GroupNorm CTAs then still fit two per SM next to them, the other order does
        # not (three resident GroupNorm CTAs hold 61 K of the SM's 64 K registers)
        side = _SIDE_STREAMS[key] = torch.cuda.Stream(E.device, priority=-1)
    side.wait_event(after)
    main_handle, E.stream = E.stream, side.cuda_stream
    try:
        fn()
    finally:
        E.stream = main_handle
    return _event_on(side)


def grad_of(p: torch.nn.Parameter) -> Optional[torch.Tensor]:
    """fp32 gradient buffer of a parameter (created zeroed on first use; kernels accumulate)."""
    if not p.requires_grad:
        return None
    if p.grad is None:
        p.grad = torch.zeros_like(p, memory_format=torch.contiguous_format)
    return p.grad


def _gptr(p) -> Optional[int]:
    g = grad_of(p) if p is not None else None
    return g.data_ptr() if g is not None else None


# ----------------------------------------------------------------------------------------------
# primitive ops (one C-ABI call each)
# ----------------------------------------------------------------------------------------------
def conv(E: Exec, x: Act, wpack: torch.Tensor, out: Act, k: int, stride: int = 1, pad: int = 0, *,
         bias: Optional[torch.Tensor] = None, tbias: Optional[torch.Tensor] = None, res: Optional[Act] = None,
         z: Optional[Act] = None, accum: bool = False, a_silu: bool = False, mode: int = _lib.CONV_NORMAL,
         dt: Optional[int] = None, in2: Optional[Act] = None, w2pack: Optional[torch.Tensor] = None, up_phase: int = 0) -> Act:
    """`in2` / `w2pack`: out = conv(x; w) + conv1x1(in2; w2) in one launch (see ddpm_conv_args.in2).
    `mode=CONV_UP2X_PHASE`, `up_phase`: one output phase of conv3x3(nearest x2 (x)) from the low-resolution x."""
    dt = x.dt if dt is None else dt
    a = _conv_args(E, x, wpack, out, k, stride, pad, bias, tbias, res, z, accum, a_silu, mode, dt, in2, w2pack, up_phase)
    _lib.call("ddpm_conv", C.byref(a), E.stream)
    return out


def _conv_args(E, x, wpack, out, k, stride, pad, bias, tbias, res, z, accum, a_silu, mode, dt, in2, w2pack, up_phase):
    a = _lib.ConvArgs()
    a.inp, a.out = x.desc(), out.desc()
    a.w = wpack.data_ptr()
    if in2 is not None:
        a.in2, a.w2 = in2.desc(), w2pack.data_ptr()
    else:
        a.in2, a.w2 = _NULL, None
    a.bias = bias.data_ptr() if bias is not None else None
    a.bias_n = bias.numel() if bias is not None else 0
    if tbias is not None:
        a.tbias, a.tbias_pitch = tbias.data_ptr(), tbias.stride(0)
    else:
        a.tbias, a.tbias_pitch = None, 0
    a.res = res.desc() if res is not None else _NULL
    a.z = z.desc() if z is not None else _NULL
    a.KH = a.KW = k
    a.stride, a.pad, a.mode = stride, pad, mode
    a.a_silu = 1 if a_silu else 0
    a.epi = (_lib.EPI_ACCUM if accum else 0) | (_lib.EPI_DSILU if z is not None else 0)
    a.dtype = dt
    a.prefer_tc = E.prefer_tc
    a.up_phase = up_phase
    return a


def wgrad(E: Exec, act: Act, dy: Act, w: torch.nn.Parameter, k: int, stride: int = 1, pad: int = 0,
          a_silu: bool = False, bias: Optional[torch.nn.Parameter] = None) -> None:
    """dW += dY^T (*) act (and db += sum_pixels dY when `bias` is given, from the same launch on the tensor-core
    path).  `act` / `dy` may carry zero-padded channels beyond the parameter's shape."""
    g = grad_of(w)
    if g is None:
        if bias is not None:
            colsum(E, dy.slice(0, bias.numel()) if dy.C != bias.numel() else dy, None, bias)
        return
    a = _lib.WgradArgs()
    a.act, a.dy = act.desc(), dy.desc()
    a.dw = g.data_ptr()
    a.KH = a.KW = k
    a.stride, a.pad = stride, pad
    a.a_silu = 1 if a_silu else 0
    a.dtype = act.dt
    a.prefer_tc = E.prefer_tc
    a.workspace, a.workspace_bytes = None, 0
    a.cin_valid = w.shape[1] if act.C != w.shape[1] else 0
    a.cout_valid = w.shape[0] if dy.C != w.shape[0] else 0
    a.dbias = _gptr(bias)
    if E.use_tc and act.dt == _lib.BF16 and stride == 1:
        need = int(_lib.lib.ddpm_wgrad_workspace_bytes(C.byref(a)))
        if need > 0:
            ws = E.workspace(need)
            a.workspace, a.workspace_bytes = ws.data_ptr(), need
    _lib.call("ddpm_conv_wgrad", C.byref(a), E.stream)


def colsum(E: Exec, dy: Act, out_nc: Optional[torch.Tensor], bias: Optional[torch.nn.Parameter]) -> None:
    gb = _gptr(bias)
    if out_nc is None and gb is None:
        return
    _lib.call("ddpm_colsum", C.byref(dy.desc()), dy.dt, out_nc.data_ptr() if out_nc is not None else None, gb, E.stream)


def gn_stats(E: Exec, x: Act, groups: int) -> torch.Tensor:
    st = torch.empty((x.N, groups, 2), dtype=torch.float64, device=E.device)
    _lib.call("ddpm_gn_stats", C.byref(x.desc()), x.dt, groups, st.data_ptr(), E.stream)
    return st


def gn_apply(E: Exec, x: Act, st: torch.Tensor, gn: torch.nn.GroupNorm, act: int, p_drop: float, layer: int,
             out: Optional[Act] = None) -> Act:
    if out is None:
        out = E.act(x.N, x.H, x.W, x.C)
    _lib.call("ddpm_gn_apply", C.byref(x.desc()), x.dt, gn.num_groups, st.data_ptr(), gn.weight.data_ptr(),
              gn.bias.data_ptr(), float(gn.eps), act, float(p_drop), E.rng.data_ptr() if p_drop > 0 else None,
              layer, C.byref(out.desc()), E.stream)
    return out


def gn_fwd(E: Exec, x: Act, gn: torch.nn.GroupNorm, act: int, p_drop: float, layer: int,
           out: Optional[Act] = None):
    """Fused stats + normalise + activation (+dropout): returns (out, stats)."""
    if out is None:
        out = E.act(x.N, x.H, x.W, x.C)
    st = torch.empty((x.N, gn.num_groups, 2), dtype=torch.float64, device=E.device)
    _lib.call("ddpm_gn_fwd", C.byref(x.desc()), x.dt, gn.num_groups, st.data_ptr(), gn.weight.data_ptr(),
              gn.bias.data_ptr(), float(gn.eps), act, float(p_drop), E.rng.data_ptr() if p_drop > 0 else None,
              layer, C.byref(out.desc()), E.stream)
    return out, st


def gn_bwd(E: Exec, x: Act, st: torch.Tensor, gn: torch.nn.GroupNorm, act: int, p_drop: float, layer: int,
           dy: Act, dx: Act, accumulate: bool, colsum_nc: Optional[torch.Tensor] = None,
           colsum_bias: Optional[torch.nn.Parameter] = None, dy_scratch: bool = False) -> Act:
    """`colsum_nc` ([N][C] fp32, overwritten) / `colsum_bias` (parameter whose .grad is accumulated) receive the
    channel sums of the final dx from the same launch.  `dy_scratch`: dy is dead after this call (true for every
    gradient temporary of the UNet backward) -> the kernel may overwrite it (see ddpm_gn_bwd_colsum)."""
    _lib.call("ddpm_gn_bwd_colsum", C.byref(x.desc()), x.dt, gn.num_groups, st.data_ptr(), gn.weight.data_ptr(),
              gn.bias.data_ptr(), float(gn.eps), act, float(p_drop), E.rng.data_ptr() if p_drop > 0 else None,
              layer, C.byref(dy.desc()), C.byref(dx.desc()), 1 if accumulate else 0, _gptr(gn.weight),
              _gptr(gn.bias), colsum_nc.data_ptr() if colsum_nc is not None else None, _gptr(colsum_bias),
              1 if dy_scratch else 0, E.stream)
    return dx


def add(E: Exec, a: Act, b: Act, out: Act) -> Act:
    _lib.call("ddpm_add", C.byref(a.desc()), C.byref(b.desc()), C.byref(out.desc()), a.dt, E.stream)
    return out


def to_nhwc(E: Exec, x: torch.Tensor, halo=1, cpad: int = 0) -> Act:
    """NCHW-shaped torch tensor (any strides, fp32/bf16) -> pooled NHWC activation (optionally with the
    channel count padded with zeros to `cpad` for the tensor-core kernels)."""
    B, Cc, H, W = x.shape
    src_dt = _lib.F32 if x.dtype == torch.float32 else _lib.BF16
    if x.dtype not in (torch.float32, torch.bfloat16):
        x = x.float()
        src_dt = _lib.F32
    out = E.act(B, H, W, max(Cc, cpad), halo)
    sn, sc, sh, sw = x.stride()
    _lib.call("ddpm_nchw_to_nhwc", x.data_ptr(), src_dt, Cc, sn, sc, sh, sw, C.byref(out.desc()), E.dt, E.stream)
    return out


def to_nchw(E: Exec, a: Act, out_dtype: torch.dtype) -> torch.Tensor:
    out = torch.empty((a.N, a.C, a.H, a.W), dtype=out_dtype, device=E.device)
    dd = _lib.F32 if out_dtype == torch.float32 else _lib.BF16
    sn, sc, sh, sw = out.stride()
    _lib.call("ddpm_nhwc_to_nchw", C.byref(a.desc()), a.dt, out.data_ptr(), dd, sn, sc, sh, sw, E.stream)
    return out


# ----------------------------------------------------------------------------------------------
# linear layers of the time path (fp32, H=W=1)
# ----------------------------------------------------------------------------------------------
def linear_fwd(E: Exec, x: torch.Tensor, lin: torch.nn.Linear, a_silu: bool) -> torch.Tensor:
    B = x.shape[0]
    wf, _ = E.wcache.get(E, lin.weight, _lib.F32, False)
    out = E.f32(B, lin.out_features)
    conv(E, E.vec(x, B, lin.in_features), wf, E.vec(out, B, lin.out_features), 1, bias=lin.bias, a_silu=a_silu, dt=_lib.F32)
    return out


def linear_bwd(E: Exec, x: torch.Tensor, lin: torch.nn.Linear, a_silu: bool, dy: torch.Tensor,
               dx: Optional[torch.Tensor], dx_accum: bool, need_dx: bool = True) -> Optional[torch.Tensor]:
    """y = lin(silu?(x)).  Accumulates dW, db; returns d/dx (multiplied by silu'(x) when a_silu)."""
    B = x.shape[0]
    xa, dya = E.vec(x, B, lin.in_features), E.vec(dy, B, lin.out_features)
    wgrad(E, xa, dya, lin.weight, 1, a_silu=a_silu)
    if lin.bias is not None and lin.bias.requires_grad:
        colsum(E, Act.wrap(dy, 1, 1, B, lin.out_features, _lib.F32, 0), None, lin.bias)
    if not need_dx:
        return None
    _, wd = E.wcache.get(E, lin.weight, _lib.F32, True)
    if dx is None:
        dx = E.f32(B, lin.in_features)
        dx_accum = False
    conv(E, dya, wd, E.vec(dx, B, lin.in_features), 1, z=xa if a_silu else None, accum=dx_accum, dt=_lib.F32)
    return dx


def time_proj_all_fwd(E: Exec, model, rbs: list, temb: torch.Tensor) -> List[torch.Tensor]:
    """Per-block time biases `time_proj(temb)` (unet_backbone.py:25-27,41) for every ResBlock with ONE launch; returns
    column-slice views [B][C_i] of one [B][sum C_i] buffer (the convolution epilogue takes a row pitch)."""
    lins = [b.time_proj[1] for b in rbs]
    # conv1's bias is folded into the time bias here (bias2), so that conv1's epilogue adds one per-image vector
    # instead of two (in situ the bias + time-bias epilogue cost 30 us of a 97 us launch at 96 ch @ 64x64)
    cb = [b.conv1.bias for b in rbs]
    sig = tuple((l.weight.data_ptr(), l.bias.data_ptr() if l.bias is not None else 0, c.data_ptr() if c is not None else 0)
                for l, c in zip(lins, cb))
    tab = getattr(model, "_ddpm_tp_table", None)
    if tab is None or tab[0] != sig or tab[1].device != temb.device:
        arr = (_lib.LinEntry * len(lins))()
        col, offs = 0, []
        for i, l in enumerate(lins):
            arr[i] = _lib.LinEntry(l.weight.data_ptr(), l.bias.data_ptr() if l.bias is not None else None, l.out_features, col,
                                   cb[i].data_ptr() if cb[i] is not None else None)
            offs.append(col)
            col += (l.out_features + 3) // 4 * 4            # 16-byte aligned slices -> float4 time-bias loads in the conv epilogue
        dev_tab = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).to(temb.device)
        tab = (sig, dev_tab, offs, col, max(l.out_features for l in lins))
        object.__setattr__(model, "_ddpm_tp_table", tab)
    _, dev_tab, offs, total, max_n = tab
    B, K = temb.shape
    out = E.f32(B, total)
    _lib.call("ddpm_linear_grouped_fwd", temb.data_ptr(), B, K, temb.stride(0), dev_tab.data_ptr(), len(lins), max_n,
              out.data_ptr(), total, 1, E.stream)
    return [out[:, o:o + l.out_features] for o, l in zip(offs, lins)]


def time_proj_bwd(E: Exec, temb: torch.Tensor, lin: torch.nn.Linear, dtb: torch.Tensor, dtemb: Optional[torch.Tensor]) -> torch.Tensor:
    """dW, db of one time_proj and the accumulated d temb in one launch."""
    B, K = temb.shape
    accum = dtemb is not None
    if dtemb is None:
        dtemb = E.f32(B, K)
    gw = grad_of(lin.weight)
    if gw is None:
        gw = torch.zeros_like(lin.weight)                   # frozen weight: gradient discarded
    _lib.call("ddpm_time_proj_bwd", temb.data_ptr(), B, K, dtb.data_ptr(), dtb.stride(0), lin.out_features,
              lin.weight.data_ptr(), gw.data_ptr(), _gptr(lin.bias), dtemb.data_ptr(), 1 if accum else 0, E.stream)
    return dtemb


# ----------------------------------------------------------------------------------------------
# ResBlock  (unet_backbone.py:10-44)
# ----------------------------------------------------------------------------------------------
def resblock_fwd(E: Exec, blk, x: Act, tbias: torch.Tensor, out: Optional[Act] = None, layer: int = 0,
                 tbias_has_b1: bool = False):
    """h = conv1(silu(gn1(x))) + b1 + tbias ; out = conv2(drop(silu(gn2(h)))) + b2 + skip(x).
    `tbias_has_b1`: the caller's time bias already contains conv1's bias (time_proj_all_fwd)."""
    Cout = blk.out_ch
    p_drop = float(blk.drop.p) if (E.training and isinstance(blk.drop, torch.nn.Dropout)) else 0.0
    a1, st1 = gn_fwd(E, x, blk.norm1, 1, 0.0, 0)
    w1, _ = E.wcache.get(E, blk.conv1.weight, E.dt, E.need_grad)
    h = conv(E, a1, w1, E.act(x.N, x.H, x.W, Cout), 3, 1, 1, bias=None if tbias_has_b1 else blk.conv1.bias, tbias=tbias)
    a2, st2 = gn_fwd(E, h, blk.norm2, 1, p_drop, layer)
    w2, _ = E.wcache.get(E, blk.conv2.weight, E.dt, E.need_grad)
    if out is None:
        out = E.act(x.N, x.H, x.W, Cout)
    if isinstance(blk.skip, torch.nn.Conv2d):
        ws, _ = E.wcache.get(E, blk.skip.weight, E.dt, E.need_grad)
        if fuse_skip_enabled() and blk.skip.bias is not None and blk.conv2.bias is not None:
            # conv2(a2) + skip(x) as ONE implicit GEMM (K = 9*Cout + Cin): no separate 1x1 launch, no read-modify-write of
            # `out`; the two biases are summed first (a 96..192-element add)
            conv(E, a2, w2, out, 3, 1, 1, bias=blk.conv2.bias.detach() + blk.skip.bias.detach(), in2=x, w2pack=ws)
        else:
            conv(E, x, ws, out, 1, bias=blk.skip.bias)
            conv(E, a2, w2, out, 3, 1, 1, bias=blk.conv2.bias, accum=True)
    else:
        conv(E, a2, w2, out, 3, 1, 1, bias=blk.conv2.bias, res=x)
    saved = (x, st1, a1, h, st2, a2, p_drop, layer) if E.need_grad else None
    return out, saved


def resblock_bwd(E: Exec, blk, saved, dout: Act, dx: Optional[Act] = None, dx_accum: bool = False):
    """Returns (dx, dtbias [B][Cout] fp32).  `dout` may be overwritten (it becomes dx when the skip
    is the identity and no explicit target is given)."""
    x, st1, a1, h, st2, a2, p_drop, layer = saved
    has_skip_conv = isinstance(blk.skip, torch.nn.Conv2d)
    if E.use_tc and overlap_enabled() and getattr(E, "overlap_ok", True):
        return _resblock_bwd_overlapped(E, blk, saved, dout, dx, dx_accum)
    # conv2 (+ skip conv) parameter gradients
    wgrad(E, a2, dout, blk.conv2.weight, 3, 1, 1, bias=blk.conv2.bias)
    _, w2d = E.wcache.get(E, blk.conv2.weight, E.dt, True)
    da2 = conv(E, dout, w2d, E.act(x.N, x.H, x.W, blk.out_ch), 3, 1, 1)
    dtb = E.f32(x.N, blk.out_ch)
    # in place (dh overwrites da2); the same launch emits d(time bias) and d(conv1.bias)
    dh = gn_bwd(E, h, st2, blk.norm2, 1, p_drop, layer, da2, da2, False, colsum_nc=dtb, colsum_bias=blk.conv1.bias,
                dy_scratch=True)
    wgrad(E, a1, dh, blk.conv1.weight, 3, 1, 1)
    _, w1d = E.wcache.get(E, blk.conv1.weight, E.dt, True)
    da1 = conv(E, dh, w1d, E.act(x.N, x.H, x.W, blk.in_ch), 3, 1, 1)
    if has_skip_conv:
        wgrad(E, x, dout, blk.skip.weight, 1, bias=blk.skip.bias)
        _, wsd = E.wcache.get(E, blk.skip.weight, E.dt, True)
        if dx is None:
            dx, dx_accum = E.act(x.N, x.H, x.W, blk.in_ch), False
        conv(E, dout, wsd, dx, 1, accum=dx_accum)
        gn_bwd(E, x, st1, blk.norm1, 1, 0.0, 0, da1, dx, True, dy_scratch=True)
    else:
        if dx is None:
            dx = gn_bwd(E, x, st1, blk.norm1, 1, 0.0, 0, da1, dout, True, dy_scratch=True)       # dout += gn_bwd -> dx
        else:
            gn_bwd(E, x, st1, blk.norm1, 1, 0.0, 0, da1, dx, dx_accum, dy_scratch=True)
            add(E, dx, dout, dx)
    return dx, dtb


def _resblock_bwd_overlapped(E: Exec, blk, saved, dout: Act, dx: Optional[Act], dx_accum: bool):
    """Same arithmetic as the serial path; the three weight-gradient launches run on the side stream, each paired
    with the GroupNorm backward that follows on the main stream:
        main:  dgrad(conv2) | gn_bwd(norm2) | dgrad(conv1) [skip dgrad] | gn_bwd(norm1)
        side:               | wgrad(conv2)[,skip]          |            | wgrad(conv1)
    Hazards: wgrad(conv2/skip) read `dout`, which gn_bwd(norm1) overwrites -> main waits for them first; wgrad(conv1)
    reads dh / a1, which go back to the buffer pool when this function returns -> main waits before returning."""
    x, st1, a1, h, st2, a2, p_drop, layer = saved
    has_skip_conv = isinstance(blk.skip, torch.nn.Conv2d)
    main = torch.cuda.current_stream(E.device)
    # gradient buffers that do not exist yet are created (zero-filled) on the MAIN stream, before the fork events
    for prm in (blk.conv2.weight, blk.conv2.bias, blk.conv1.weight) + ((blk.skip.weight, blk.skip.bias) if has_skip_conv else ()):
        if prm is not None:
            grad_of(prm)
    _, w2d = E.wcache.get(E, blk.conv2.weight, E.dt, True)
    da2 = conv(E, dout, w2d, E.act(x.N, x.H, x.W, blk.out_ch), 3, 1, 1)

    def side1():
        wgrad(E, a2, dout, blk.conv2.weight, 3, 1, 1, bias=blk.conv2.bias)
        if has_skip_conv:
            wgrad(E, x, dout, blk.skip.weight, 1, bias=blk.skip.bias)
    s1 = wgrad_async(E, _event_on(main), side1)
    dtb = E.f32(x.N, blk.out_ch)
    dh = gn_bwd(E, h, st2, blk.norm2, 1, p_drop, layer, da2, da2, False, colsum_nc=dtb, colsum_bias=blk.conv1.bias,
                dy_scratch=True)
    _, w1d = E.wcache.get(E, blk.conv1.weight, E.dt, True)
    da1 = conv(E, dh, w1d, E.act(x.N, x.H, x.W, blk.in_ch), 3, 1, 1)
    if has_skip_conv:
        _, wsd = E.wcache.get(E, blk.skip.weight, E.dt, True)
        if dx is None:
            dx, dx_accum = E.act(x.N, x.H, x.W, blk.in_ch), False
        conv(E, dout, wsd, dx, 1, accum=dx_accum)
    s2 = wgrad_async(E, _event_on(main), lambda: wgrad(E, a1, dh, blk.conv1.weight, 3, 1, 1))
    main.wait_event(s1)                                   # dout is about to be overwritten / handed on
    if has_skip_conv:
        gn_bwd(E, x, st1, blk.norm1, 1, 0.0, 0, da1, dx, True, dy_scratch=True)
    else:
        if dx is None:
            dx = gn_bwd(E, x, st1, blk.norm1, 1, 0.0, 0, da1, dout, True, dy_scratch=True)       # dout += gn_bwd -> dx
        else:
            gn_bwd(E, x, st1, blk.norm1, 1, 0.0, 0, da1, dx, dx_accum, dy_scratch=True)
            add(E, dx, dout, dx)
    main.wait_event(s2)                                   # dh / a1 / a2 are recycled by the caller from here on
    return dx, dtb


# ----------------------------------------------------------------------------------------------
# AttnBlock  (attention.py:42-74)
# ----------------------------------------------------------------------------------------------
def attn_fwd(E: Exec, blk, x: Act, out: Optional[Act] = None):
    heads, d = blk.num_heads, blk.head_dim
    inner = heads * d
    wq, _ = E.wcache.get(E, blk.qkv.weight, E.dt, E.need_grad)
    a, st = gn_fwd(E, x, blk.norm, 0, 0.0, 0)
    qkv = conv(E, a, wq, E.act(x.N, x.H, x.W, 3 * inner), 1)
    o = E.act(x.N, x.H, x.W, inner)
    lse = E.f32(x.N, heads, x.H * x.W)
    _lib.call("ddpm_attn_fwd", C.byref(qkv.desc()), C.byref(o.desc()), heads, d, lse.data_ptr(), E.dt, E.stream)
    wp, _ = E.wcache.get(E, blk.proj.weight, E.dt, E.need_grad)
    if out is None:
        out = E.act(x.N, x.H, x.W, x.C)
    conv(E, o, wp, out, 1, bias=blk.proj.bias, res=x)
    saved = (x, st, a, qkv, o, lse) if E.need_grad else None
    return out, saved


def attn_bwd(E: Exec, blk, saved, dout: Act, dx: Optional[Act] = None, dx_accum: bool = False) -> Act:
    x, st, a, qkv, o, lse = saved
    heads, d = blk.num_heads, blk.head_dim
    inner = heads * d
    n_tok = x.H * x.W
    wgrad(E, o, dout, blk.proj.weight, 1, bias=blk.proj.bias)
    _, wpd = E.wcache.get(E, blk.proj.weight, E.dt, True)
    do = conv(E, dout, wpd, E.act(x.N, x.H, x.W, inner), 1)
    dqkv = E.act(x.N, x.H, x.W, 3 * inner)
    # N x N scratch only on the CUDA-core path; the tcgen05 backward recomputes P from lse and needs one float per query
    need = int(_lib.lib.ddpm_attn_bwd_scratch_floats(C.byref(qkv.desc()), C.byref(o.desc()), heads, d, E.dt))
    scratch = E.f32(max(need, 1))
    _lib.call("ddpm_attn_bwd", C.byref(qkv.desc()), C.byref(o.desc()), C.byref(do.desc()), lse.data_ptr(),
              C.byref(dqkv.desc()), heads, d, scratch.data_ptr(), E.dt, E.stream)
    wgrad(E, a, dqkv, blk.qkv.weight, 1)
    _, wqd = E.wcache.get(E, blk.qkv.weight, E.dt, True)
    da = conv(E, dqkv, wqd, E.act(x.N, x.H, x.W, x.C), 1)
    if dx is None:
        return gn_bwd(E, x, st, blk.norm, 0, 0.0, 0, da, dout, True, dy_scratch=True)
    gn_bwd(E, x, st, blk.norm, 0, 0.0, 0, da, dx, dx_accum, dy_scratch=True)
    return add(E, dx, dout, dx)


# ----------------------------------------------------------------------------------------------
# Downsample / Upsample  (unet_backbone.py:47-64)
# ----------------------------------------------------------------------------------------------
def down_fwd(E: Exec, mod, x: Act, out: Optional[Act] = None):
    w, _ = E.wcache.get(E, mod.conv.weight, E.dt, E.need_grad)
    Ho, Wo = (x.H - 1) // 2 + 1, (x.W - 1) // 2 + 1
    if out is None:
        out = E.act(x.N, Ho, Wo, x.C)
    conv(E, x, w, out, 3, 2, 1, bias=mod.conv.bias)
    return out, (x if E.need_grad else None)


def down_bwd(E: Exec, mod, saved, dout: Act, dx: Optional[Act], dx_accum: bool) -> Act:
    x = saved
    _, wd = E.wcache.get(E, mod.conv.weight, E.dt, True)
    if dx is None:
        dx, dx_accum = E.act(x.N, x.H, x.W, x.C), False
    if E.use_tc and x.H % 2 == 0 and x.W % 2 == 0:
        # stride-2 gradients as stride-1 tensor-core problems on the zero-interleaved dY
        up = E.act(x.N, x.H, x.W, dout.C)
        _lib.call("ddpm_zero_upsample2x", C.byref(dout.desc()), C.byref(up.desc()), E.dt, E.stream)
        wgrad(E, x, up, mod.conv.weight, 3, 1, 1, bias=mod.conv.bias)        # zeros of `up` add nothing to the bias sum
        conv(E, up, wd, dx, 3, 1, 1, accum=dx_accum)
    else:
        wgrad(E, x, dout, mod.conv.weight, 3, 2, 1, bias=mod.conv.bias)
        conv(E, dout, wd, dx, 3, 2, 1, accum=dx_accum, mode=_lib.CONV_TRANSPOSED)
    return dx


def fold_upsample_enabled() -> bool:
    import os
    return os.environ.get("DDPM_B200_FOLD_UPSAMPLE", "1") != "0"


def up_fwd(E: Exec, mod, x: Act, out: Optional[Act] = None):
    """nearest x2 + conv3x3 (unet_backbone.py:56-64).  On the tensor-core path the up-sampling is folded into the
    convolution: each of the four output phases (2y+py, 2x+px) is a 2x2-tap convolution of the LOW-resolution input with
    pre-summed weights -- 16 instead of 36 multiply-adds per output quad, and the 4x larger up-sampled tensor is never
    written.  Used when no gradient is needed (sampling: DDIM-100 374 -> 393 samples/s); with gradients the
    up-sampled tensor has to exist for the weight / data gradients and folding the forward alone measured no gain
    (12.08 vs 12.02 ms per step), so training keeps the single 3x3 launch."""
    cout = mod.conv.out_channels
    fold = (E.use_tc and not E.need_grad and fold_upsample_enabled() and x.C % 16 == 0 and cout % 16 == 0
            and x.W + 2 <= 300 and x.pitch % 8 == 0 and x.halo == 1)
    u = None
    if E.need_grad or not fold:
        u = E.act(x.N, 2 * x.H, 2 * x.W, x.C)
        _lib.call("ddpm_upsample2x", C.byref(x.desc()), C.byref(u.desc()), E.dt, E.stream)
    if out is None:
        out = E.act(x.N, 2 * x.H, 2 * x.W, cout)
    if fold:
        wp = E.wcache.get_up2x(E, mod.conv.weight, E.dt)
        for ph in range(4):
            conv(E, x, wp[ph], out, 2, 1, 0, bias=mod.conv.bias, mode=_lib.CONV_UP2X_PHASE, up_phase=ph)
    else:
        w, _ = E.wcache.get(E, mod.conv.weight, E.dt, E.need_grad)
        conv(E, u, w, out, 3, 1, 1, bias=mod.conv.bias)
    return out, (u if E.need_grad else None)


def up_bwd(E: Exec, mod, saved, dout: Act, dx: Optional[Act] = None, dx_accum: bool = False) -> Act:
    u = saved
    wgrad(E, u, dout, mod.conv.weight, 3, 1, 1, bias=mod.conv.bias)
    _, wd = E.wcache.get(E, mod.conv.weight, E.dt, True)
    du = conv(E, dout, wd, E.act(u.N, u.H, u.W, u.C), 3, 1, 1)
    if dx is None:
        dx, dx_accum = E.act(u.N, u.H // 2, u.W // 2, u.C), False
    _lib.call("ddpm_upsample2x_bwd", C.byref(du.desc()), C.byref(dx.desc()), E.dt, 1 if dx_accum else 0, E.stream)
    return dx


# ----------------------------------------------------------------------------------------------
# time path  (attention.py:7-35, unet_backbone.py:25-27)
# ----------------------------------------------------------------------------------------------
def sinusoid(E: Exec, t: torch.Tensor, dim: int) -> torch.Tensor:
    B = t.shape[0]
    if t.dtype == torch.int64:
        isf = 0
    else:
        t = t.float()
        isf = 1
    t = t.contiguous()
    out = E.f32(B, dim)
    _lib.call("ddpm_sinusoid", t.data_ptr(), isf, B, dim, out.data_ptr(), _lib.F32, E.stream)
    return out


def time_mlp_fwd(E: Exec, mlp, e0: torch.Tensor):
    h1 = linear_fwd(E, e0, mlp.net[0], False)
    temb = linear_fwd(E, h1, mlp.net[2], True)
    return temb, ((e0, h1) if E.need_grad else None)


def time_mlp_bwd(E: Exec, mlp, saved, dtemb: torch.Tensor, need_dx: bool = False):
    e0, h1 = saved
    dh1 = linear_bwd(E, h1, mlp.net[2], True, dtemb, None, False)
    return linear_bwd(E, e0, mlp.net[0], False, dh1, None, False, need_dx=need_dx)


# ----------------------------------------------------------------------------------------------
# UNetDenoiser forward / backward  (unet_backbone.py:166-216)
# ----------------------------------------------------------------------------------------------
def _is_res(m) -> bool:
    return hasattr(m, "conv1") and hasattr(m, "time_proj")


def _is_attn(m) -> bool:
    return hasattr(m, "qkv") and hasattr(m, "proj")


def unet_resblocks(model) -> list:
    """All ResBlocks in forward order (dropout layer ids / time_proj order)."""
    out = []
    for down in model.downs:
        out += [b for b in down.blocks if _is_res(b)]
    out += [b for b in model.mid if _is_res(b)]
    for up in model.ups:
        out += [b for b in up.blocks if _is_res(b)]
    return out


def unet_forward(E: Exec, model, x: torch.Tensor, t: torch.Tensor, out_dtype: torch.dtype):
    """Returns (eps_pred NCHW tensor, saved-state for unet_backward or None)."""
    B, Cin, H, W = x.shape
    L = len(model.downs)
    if H % (1 << (L - 1)) or W % (1 << (L - 1)):
        raise NotImplementedError(
            f"ddpm_b200 UNet needs H, W divisible by {1 << (L - 1)} (got {H}x{W}); the reference's "
            "nearest-resize of mismatched skips (unet_backbone.py:202-203) is not implemented")
    rbs = unet_resblocks(model)
    rb_index = {id(b): i for i, b in enumerate(rbs)}
    tape: list = []
    G = E.need_grad

    # ---- time path: temb, then one fp32 [B][Cout] bias per ResBlock
    e0 = sinusoid(E, t, model.time_pos_emb.dim)
    temb, mlp_saved = time_mlp_fwd(E, model.time_mlp, e0)
    tbs = time_proj_all_fwd(E, model, rbs, temb) if rbs else []

    # ---- concat buffers, one per decoder level: [cur | skip]
    enc_out_ch = []
    for down in model.downs:
        last = [b for b in down.blocks][-1]
        enc_out_ch.append(last.out_ch if _is_res(last) else last.channels)
    cats = []
    for j, up in enumerate(model.ups):
        lvl = L - 1 - j
        first = up.blocks[0]
        cat_c = first.in_ch
        sk = enc_out_ch[lvl]
        cats.append(E.act(B, H >> lvl, W >> lvl, cat_c))
        assert cat_c - sk > 0
    cur_ch_of = [cats[j].C - enc_out_ch[L - 1 - j] for j in range(L)]

    # ---- encoder
    cpad = 16 if E.use_tc else 0                       # tcgen05 K-chunk / N granularity
    x_in = to_nhwc(E, x, cpad=cpad)
    w_in, _ = E.wcache.get(E, model.in_conv.weight, E.dt, False, cin_pad=cpad)
    cur = conv(E, x_in, w_in, E.act(B, H, W, model.in_conv.out_channels), 3, 1, 1, bias=model.in_conv.bias)
    if G:
        tape.append(("in", x_in))
    for li, down in enumerate(model.downs):
        j = L - 1 - li
        blocks = list(down.blocks)
        for bi, blk in enumerate(blocks):
            tgt = cats[j].slice(cur_ch_of[j], enc_out_ch[li]) if bi == len(blocks) - 1 else None
            if _is_res(blk):
                i = rb_index[id(blk)]
                cur, sv = resblock_fwd(E, blk, cur, tbs[i], tgt, i + 1, True)
                if G:
                    tape.append(("res", blk, sv, i))
            else:
                cur, sv = attn_fwd(E, blk, cur, tgt)
                if G:
                    tape.append(("attn", blk, sv))
        if G:
            tape.append(("skip", j))
        if not isinstance(down.down, torch.nn.Identity):
            cur, sv = down_fwd(E, down.down, cur)
            if G:
                tape.append(("down", down.down, sv))

    # ---- bottleneck
    mids = [m for m in model.mid if not isinstance(m, torch.nn.Identity)]
    for mi, blk in enumerate(mids):
        tgt = cats[0].slice(0, cur_ch_of[0]) if (mi == len(mids) - 1 and isinstance(model.ups[0].up, torch.nn.Identity)) else None
        if _is_res(blk):
            i = rb_index[id(blk)]
            cur, sv = resblock_fwd(E, blk, cur, tbs[i], tgt, i + 1, True)
            if G:
                tape.append(("res", blk, sv, i))
        else:
            cur, sv = attn_fwd(E, blk, cur, tgt)
            if G:
                tape.append(("attn", blk, sv))

    # ---- decoder
    for j, up in enumerate(model.ups):
        if not isinstance(up.up, torch.nn.Identity):
            cur, sv = up_fwd(E, up.up, cur, cats[j].slice(0, cur_ch_of[j]))
            if G:
                tape.append(("up", up.up, sv))
        elif j != 0:
            raise NotImplementedError("Identity up-sampler below the first decoder level")
        cur = cats[j]
        if G:
            tape.append(("cat", j))
        for blk in up.blocks:
            i = rb_index[id(blk)]
            cur, sv = resblock_fwd(E, blk, cur, tbs[i], None, i + 1, True)
            if G:
                tape.append(("res", blk, sv, i))

    # ---- head
    w_out, _ = E.wcache.get(E, model.out_conv.weight, E.dt, G, cout_pad=cpad)
    oc = model.out_conv.out_channels
    a, st = gn_fwd(E, cur, model.out_norm, 1, 0.0, 0)
    y = conv(E, a, w_out, E.act(B, H, W, max(oc, cpad)), 3, 1, 1, bias=model.out_conv.bias)
    out = to_nchw(E, y.slice(0, oc) if y.C != oc else y, out_dtype)
    saved = None
    if G:
        saved = dict(tape=tape, head=(cur, st, a), temb=temb, mlp=mlp_saved, rbs=rbs, cats_shape=[(c.N, c.H, c.W, c.C) for c in cats],
                     cur_ch_of=cur_ch_of, enc_out_ch=enc_out_ch, L=L, xshape=tuple(x.shape))
    return out, saved


def unet_backward(E: Exec, model, saved, dy: torch.Tensor, need_dx: bool, progress=None) -> Optional[torch.Tensor]:
    """Accumulates every parameter gradient into `.grad`; returns d/dx (NCHW fp32) if requested.
    `progress(module)` is called each time all gradients of a sub-module are final (used by the
    data-parallel gradient buckets to overlap the all-reduce with the rest of backward)."""
    if progress is None:
        progress = getattr(model, "_ddpm_grad_progress", None)
    tape = saved["tape"]
    cur_h, st, a = saved["head"]
    L = saved["L"]
    B = saved["xshape"][0]
    # The weight-gradient side stream pays when kernels are short (64 px, B=128: 12.10 vs 12.21 ms per step); with the long
    # kernels of the 256-px model it only adds contention (CelebA256, B=32: 474 vs 486 img/s over five runs each).
    E.overlap_ok = B * saved["xshape"][2] * saved["xshape"][3] <= (1 << 20)
    rbs = saved["rbs"]
    dtemb: Optional[torch.Tensor] = None
    temb = saved["temb"]

    # ---- head
    cpad = 16 if E.use_tc else 0
    oc = model.out_conv.out_channels
    dyn = to_nhwc(E, dy, cpad=cpad)
    wgrad(E, a, dyn, model.out_conv.weight, 3, 1, 1, bias=model.out_conv.bias)
    _, wd = E.wcache.get(E, model.out_conv.weight, E.dt, True, cout_pad=cpad)
    da = conv(E, dyn, wd, E.act(a.N, a.H, a.W, a.C), 3, 1, 1)
    dcur = gn_bwd(E, cur_h, st, model.out_norm, 1, 0.0, 0, da, da, False, dy_scratch=True)
    del da, dyn
    if progress is not None:
        progress(model.out_conv)

    dcats: List[Optional[Act]] = [None] * L
    dx = None
    for idx in range(len(tape) - 1, -1, -1):
        ent = tape[idx]
        kind = ent[0]
        if kind == "res":
            _, blk, sv, i = ent
            dcur, dtb = resblock_bwd(E, blk, sv, dcur)
            dtemb = time_proj_bwd(E, temb, blk.time_proj[1], dtb, dtemb)
            if progress is not None:
                progress(blk)
        elif kind == "attn":
            _, blk, sv = ent
            dcur = attn_bwd(E, blk, sv, dcur)
            if progress is not None:
                progress(blk)
        elif kind == "cat":
            j = ent[1]
            # dcur is the gradient of the whole [cur | skip] buffer
            dcats[j] = dcur
            dcur = dcur.slice(0, saved["cur_ch_of"][j])
        elif kind == "up":
            _, mod, sv = ent
            dcur = up_bwd(E, mod, sv, dcur)
            if progress is not None:
                progress(mod)
        elif kind == "down":
            _, mod, sv = ent
            # gradient of the level output = skip part of dcat (+)= dgrad of the stride-2 conv
            assert tape[idx - 1][0] == "skip"
            j = tape[idx - 1][1]        # decoder level fed by this encoder level's output
            tgt = dcats[j].slice(saved["cur_ch_of"][j], saved["enc_out_ch"][L - 1 - j])
            dcur = down_bwd(E, mod, sv, dcur, tgt, True)
            if progress is not None:
                progress(mod)
        elif kind == "skip":
            j = ent[1]
            tgt = dcats[j].slice(saved["cur_ch_of"][j], saved["enc_out_ch"][L - 1 - j])
            if not _same_view(dcur, tgt):
                # last encoder level: its consumer was the bottleneck, whose dx is in `dcur`
                dcur = add(E, dcur, tgt, tgt)
        elif kind == "in":
            x_in = ent[1]
            wgrad(E, x_in, dcur, model.in_conv.weight, 3, 1, 1, bias=model.in_conv.bias)
            if need_dx:
                _, wdi = E.wcache.get(E, model.in_conv.weight, E.dt, True, cin_pad=cpad)
                dxa = conv(E, dcur, wdi, E.act(x_in.N, x_in.H, x_in.W, x_in.C), 3, 1, 1)
                ic = model.in_conv.in_channels
                dx = to_nchw(E, dxa.slice(0, ic) if dxa.C != ic else dxa, torch.float32)
    # ---- time path (the per-block time_proj gradients were produced inside the loop)
    if dtemb is not None:
        time_mlp_bwd(E, model.time_mlp, saved["mlp"], dtemb)
    if progress is not None:
        progress(None)           # everything is final
    return dx if need_dx else None


def _same_view(a: Act, b: Act) -> bool:
    return a.buf is b.buf and a.c0 == b.c0 and a.C == b.C

