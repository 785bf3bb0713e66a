"""ctypes binding of libddpm_b200.so (the C ABI declared in include/ddpm_b200.h).

There is NO fallback: if the shared library is missing and cannot be built, importing this module
raises; every wrapper raises RuntimeError on a non-zero return code.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

F32, BF16, F16 = 0, 1, 2
CLAMP_X0, DYN_THRESH = 1, 2
CONV_NORMAL, CONV_TRANSPOSED, CONV_UP2X_PHASE = 0, 1, 2
EPI_ACCUM, EPI_DSILU = 1, 2


class Tensor(C.Structure):
    """struct ddpm_tensor"""
    _fields_ = [("ptr", C.c_void_p), ("N", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
                ("C", C.c_int32), ("pitch", C.c_int32), ("halo", C.c_int32)]


class ConvArgs(C.Structure):
    """struct ddpm_conv_args"""
    _fields_ = [("inp", Tensor), ("out", Tensor), ("w", C.c_void_p), ("bias", C.c_void_p),
                ("tbias", C.c_void_p), ("tbias_pitch", C.c_int32), ("res", Tensor), ("z", Tensor),
                ("KH", C.c_int32), ("KW", C.c_int32), ("stride", C.c_int32), ("pad", C.c_int32),
                ("mode", C.c_int32), ("a_silu", C.c_int32), ("epi", C.c_int32), ("dtype", C.c_int32),
                ("prefer_tc", C.c_int32), ("bias_n", C.c_int32), ("in2", Tensor), ("w2", C.c_void_p),
                ("up_phase", C.c_int32)]


class WgradArgs(C.Structure):
    """struct ddpm_wgrad_args"""
    _fields_ = [("act", Tensor), ("dy", Tensor), ("dw", C.c_void_p), ("KH", C.c_int32),
                ("KW", C.c_int32), ("stride", C.c_int32), ("pad", C.c_int32), ("a_silu", C.c_int32),
                ("dtype", C.c_int32), ("prefer_tc", C.c_int32), ("workspace", C.c_void_p),
                ("workspace_bytes", C.c_int64), ("cin_valid", C.c_int32), ("cout_valid", C.c_int32),
                ("dbias", C.c_void_p)]


class PackEntry(C.Structure):
    """struct ddpm_pack_entry"""
    _fields_ = [("w", C.c_void_p), ("wf", C.c_void_p), ("wd", C.c_void_p), ("Cout", C.c_int32), ("Cin", C.c_int32),
                ("taps", C.c_int32), ("CiP", C.c_int32), ("CoP", C.c_int32), ("dtype", C.c_int32)]


class LinEntry(C.Structure):
    """struct ddpm_lin_entry"""
    _fields_ = [("w", C.c_void_p), ("bias", C.c_void_p), ("N", C.c_int32), ("col0", C.c_int32), ("bias2", C.c_void_p)]


class AdamHyper(C.Structure):
    """struct ddpm_adam_hyper"""
    _fields_ = [("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float),
                ("weight_decay", C.c_float), ("max_norm", C.c_float), ("ema_decay", C.c_float),
                ("adamw", C.c_int32)]


_vp, _i, _i64, _f, _u32 = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_uint32
_TP = C.POINTER(Tensor)

# name -> argtypes (restype is int except where noted); mirrors include/ddpm_b200.h one to one
SIGNATURES = {
    "ddpm_abi_version": [],
    "ddpm_num_sms": [_i, C.POINTER(C.c_int)],
    "ddpm_launch_count": [_i],
    "ddpm_launch_count_add": [_i64],
    "ddpm_schedule_create": [_vp, _i, _i, C.POINTER(_vp)],
    "ddpm_schedule_destroy": [_vp],
    "ddpm_q_sample": [_vp, _vp, _vp, _vp, _vp, _i, _i64, _vp],
    "ddpm_mse_fwd": [_vp, _i, _vp, _vp, _vp, _i, _i64, _vp],
    "ddpm_mse_bwd": [_vp, _i, _vp, _vp, _vp, _vp, _i, _i64, _vp],
    "ddpm_x0_absmax": [_vp, _vp, _vp, _i, _vp, _vp, _i, _i64, _vp],
    "ddpm_p_sample_step": [_vp, _vp, _vp, _i, _vp, _vp, _vp, _f, _i, _vp, _i, _i64, _vp],
    "ddpm_ddim_step": [_vp, _vp, _vp, _i, _vp, _vp, _vp, _f, _vp, _f, _i, _vp, _i, _i64, _vp],
    "ddpm_to_image01": [_vp, _vp, _i64, _vp],
    "ddpm_image_grid": [_vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp],
    "ddpm_batch_from_u8": [_vp, _i64, _vp, _i, _i, _i, _vp, _vp],
    "ddpm_nchw_to_nhwc": [_vp, _i, _i, _i64, _i64, _i64, _i64, _TP, _i, _vp],
    "ddpm_nhwc_to_nchw": [_TP, _i, _vp, _i, _i64, _i64, _i64, _i64, _vp],
    "ddpm_sinusoid": [_vp, _i, _i, _i, _vp, _i, _vp],
    "ddpm_gn_stats": [_TP, _i, _i, _vp, _vp],
    "ddpm_gn_apply": [_TP, _i, _i, _vp, _vp, _vp, _f, _i, _f, _vp, _u32, _TP, _vp],
    "ddpm_gn_fwd": [_TP, _i, _i, _vp, _vp, _vp, _f, _i, _f, _vp, _u32, _TP, _vp],
    "ddpm_gn_bwd": [_TP, _i, _i, _vp, _vp, _vp, _f, _i, _f, _vp, _u32, _TP, _TP, _i, _vp, _vp, _vp, _vp],
    "ddpm_gn_bwd_colsum": [_TP, _i, _i, _vp, _vp, _vp, _f, _i, _f, _vp, _u32, _TP, _TP, _i, _vp, _vp, _vp, _vp, _i, _vp],
    "ddpm_upsample2x": [_TP, _TP, _i, _vp],
    "ddpm_upsample2x_bwd": [_TP, _TP, _i, _i, _vp],
    "ddpm_zero_upsample2x": [_TP, _TP, _i, _vp],
    "ddpm_add": [_TP, _TP, _TP, _i, _vp],
    "ddpm_colsum": [_TP, _i, _vp, _vp, _vp],
    "ddpm_conv": [C.POINTER(ConvArgs), _vp],
    "ddpm_conv_wgrad": [C.POINTER(WgradArgs), _vp],
    "ddpm_wgrad_workspace_bytes": [C.POINTER(WgradArgs)],
    "ddpm_pack_weights": [_vp, _i, _i, _i, _i, _vp, _vp, _i, _i, _i, _vp],
    "ddpm_pack_weights_batched": [_vp, _i, _vp],
    "ddpm_pack_weights_up2x": [_vp, _i, _i, _vp, _i, _vp],
    "ddpm_linear_grouped_fwd": [_vp, _i, _i, _i, _vp, _i, _i, _vp, _i, _i, _vp],
    "ddpm_time_proj_bwd": [_vp, _i, _i, _vp, _i, _i, _vp, _vp, _vp, _vp, _i, _vp],
    "ddpm_attn_fwd": [_TP, _TP, _i, _i, _vp, _i, _vp],
    "ddpm_attn_bwd": [_TP, _TP, _TP, _vp, _TP, _i, _i, _vp, _i, _vp],
    "ddpm_attn_bwd_scratch_floats": [_TP, _TP, _i, _i, _i],
    "ddpm_param_reduce": [_vp, _i64, _vp, _vp],
    "ddpm_param_update": [_vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, C.POINTER(AdamHyper), _vp],
    "ddpm_scaler_update": [_vp, _vp, _vp, _f, _f, _i, _vp],
    "ddpm_grad_unscale_clip": [_vp, _i64, _vp, _vp, _f, _vp],
    "ddpm_ema_update": [_vp, _vp, _i64, _f, _vp],
    "ddpm_rng_advance": [_vp, _vp],
    "ddpm_set_force_simt": [_i],
    "ddpm_set_tc_mode": [_i, _i],
    "ddpm_abi_struct_sizes": [_vp, _i],
}


def _load() -> C.CDLL:
    path = _build.LIB
    if not os.path.exists(path) or (os.environ.get("DDPM_B200_REBUILD") == "1"):
        path = _build.build()          # raises if nvcc is missing or the build fails
    if os.environ.get("DDPM_B200_LIB"):                 # A/B measurements against another build of the same ABI
        path = os.environ["DDPM_B200_LIB"]
    lib = C.CDLL(path)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)        # AttributeError if the ABI symbol is missing
        fn.argtypes = argtypes
        fn.restype = C.c_int64 if name in ("ddpm_launch_count", "ddpm_wgrad_workspace_bytes", "ddpm_attn_bwd_scratch_floats") else C.c_int
    # the ctypes mirrors above must have exactly the layouts the library was compiled with (a silent mismatch would
    # corrupt every launch): compare sizeof() struct by struct and refuse to load otherwise
    mine = [("ddpm_tensor", Tensor), ("ddpm_conv_args", ConvArgs), ("ddpm_lin_entry", LinEntry), ("ddpm_wgrad_args", WgradArgs),
            ("ddpm_pack_entry", PackEntry), ("ddpm_adam_hyper", AdamHyper)]
    got = (C.c_int32 * len(mine))()
    n = lib.ddpm_abi_struct_sizes(got, len(mine))
    bad = [(nm, C.sizeof(t), int(got[i])) for i, (nm, t) in enumerate(mine) if i >= n or C.sizeof(t) != int(got[i])]
    if bad:
        raise ImportError(f"ddpm_b200: ABI struct layout mismatch between _lib.py and {path}: {bad} (rebuild: python __graft_entry__.py)")
    return lib


LIB_PATH = _build.LIB
lib = _load()

_CUDA_ERR = {2: "CUDA out of memory", 700: "illegal memory access", 701: "launch out of resources",
             719: "launch failure", 9: "invalid configuration", 1: "invalid value"}


def check(rc: int, name: str) -> None:
    if rc == 0:
        return
    if rc < 0:
        raise RuntimeError(f"ddpm_b200: {name} rejected its arguments (code {rc})")
    raise RuntimeError(f"ddpm_b200: {name} failed with cudaError {rc} ({_CUDA_ERR.get(rc, 'see cuda_runtime_api.h')})")


def call(name: str, *args) -> None:
    check(getattr(lib, name)(*args), name)


def stream_for(device) -> int:
    """Current CUDA stream handle of `device` for a C-ABI call.  The entry points launch on the process's CURRENT
    device (kernels, the constant-bank uploads of the schedule tables, memsets), so tensors on another GPU would be
    processed by the wrong device's kernels -- torch ops guard against that, a plain C ABI cannot.  Refuse loudly."""
    import torch
    idx = device.index if getattr(device, "index", None) is not None else torch.cuda.current_device()
    cur = torch.cuda.current_device()
    if idx != cur:
        raise RuntimeError(f"ddpm_b200: tensors live on cuda:{idx} but the current device is cuda:{cur}; call "
                           f"torch.cuda.set_device({idx}) (or use `with torch.cuda.device({idx}):`) before using the model")
    return torch.cuda.current_stream(device).cuda_stream


def launch_count(reset: bool = False) -> int:
    return int(lib.ddpm_launch_count(1 if reset else 0))
