"""Tensor-core convolution (conv_tc2_kernel) and weight gradient (wgrad_tc_kernel / wgrad_tc2_kernel + wgrad_reduce_kernel)
against a float64 reference, element by element and work unit by work unit, in every launch plan the host planners of
csrc/conv_tc.cu choose.

Reference.  The fp64 result is computed on the GPU (torch.float64) from the exact bf16 operands the kernel reads: the
activation interior, the bf16-rounded weight (flipped and transposed for the data gradient, as the weight cache packs it;
the packed copy is checked bit for bit against that), the fp32 bias and per-image time bias, the bf16 residual and the
accumulate target.  A few hundred output elements of it are recomputed as explicit dot products on the CPU, so the
reference does not rest on one library.  `A` is the same operation on absolute values (|x| * |w|, plus |bias| + |tbias| +
|res| + |acc|), the scale of every rounding error.

Error model and the three checks every case passes:
  1. Per element, a bound that cannot flake.  The tensor core multiplies bf16 operands exactly and accumulates in fp32;
     with K terms per output the accumulation error is at most K * u * A.  IEEE round-to-nearest would give u = 2^-24;
     we take u = 2^-22 because the tensor core's fp32 accumulation is not IEEE (operands are aligned to the largest
     exponent of a group and the low bits are truncated, not rounded), and a bound that has to hold for every element
     of every run needs that margin.  E = K * 2^-22 * A.
       fp32 outputs (dW, dbias):  |got - ref| <= E
       bf16 outputs:              |got - ref| <= 2^-8 * (|ref| + E) + E
     bf16 keeps 8 significant bits, so rounding to nearest moves a value by up to 2^-8 of itself (a value just above a
     power of two, half-way between two bf16 neighbours, does reach it: test_bf16_rounding_reaches_2_to_the_minus_8).
     This check catches gross local errors: a wrong pixel, a wrong channel, a stale tile.
  2. Per work unit, a tight statistical bound.  Outputs are grouped the way the kernel produces them -- a 128-pixel
     row block of padded-linear Q times one channel tile for the convolution; one (co tile, ci tile, tap) block for the
     weight gradient; one channel for the bias gradient (wgrad_reduce_kernel sums one channel per warp).
       bf16 outputs:  rms(got - ref) <= 2^-8 * rms(ref)   (pure bf16 rounding gives about a third of that)
       fp32 outputs:  rms(got - ref) <= 2^-18 * rms(A)    (split-K fp32 sums give ~2^-23)
     A failure names the worst unit and the launch plan.
  3. Bit-exact side conditions: the zero halo stays zero; when `out` is a channel slice of a wider buffer filled with a
     sentinel, the channels outside the slice keep their bits; the packed weights equal the rounded parameter.

The CPU tests at the bottom act on fp64 data only and show that these tolerances have teeth: each builds a plausible
wrong result (a lost K-chunk, a dropped or doubled pixel stage, a lost border tap, a short bias channel) and asserts that
the criteria reject it -- and records that the norm-relative 1e-2 check of test_gpu_tc.py accepts the first three.

Plans.  conv_plan / wg_plan below transcribe the launch planning of conv_tc_launch and wg_plan / wg_pair.  The weight
gradient transcription is pinned to the library's own ddpm_wgrad_workspace_bytes on the CPU; on the GPU each case checks
the kernel template and grid the planner actually launched (torch.profiler) against the transcription.  A CPU test
asserts that the case lists reach every planner regime.
"""
import ctypes as C
import json
import math
import os
import tempfile

import pytest
import torch
import torch.nn.functional as F

U_ACC = 2.0 ** -22          # fp32 accumulation on the tensor core, with a 4x margin over IEEE (see above)
U_BF16 = 2.0 ** -8          # bf16 unit round-off
RMS_BF16 = 2.0 ** -8        # criterion 2, bf16 outputs: rms(err) <= RMS_BF16 * rms(ref)
RMS_F32 = 2.0 ** -18        # criterion 2, fp32 outputs: rms(err) <= RMS_F32 * rms(A)
DEFAULT_SMS = 148


def sm_count():
    if torch.cuda.is_available():
        return torch.cuda.get_device_properties(0).multi_processor_count
    return DEFAULT_SMS


def cdiv(a, b):
    return -(-a // b)


# ================================================================================================================
# planner transcriptions (csrc/conv_tc.cu)
# ================================================================================================================
def pick_nt(cout):                                   # conv_tc.cu pick_nt
    if cout <= 256:
        return cout
    for nt in range(256, 63, -16):
        if cout % nt == 0:
            return nt
    return 0


def conv_plan(cin, cout, N, H, W, taps, kch2=0, sub=False, up=False, flags=0, sms=None, v256_ok=True,
              bias_aligned=True, tbias_vec=True):
    """conv_tc_launch: H, W, N are the geometry of the kernel's input operand (the low-resolution input for `up`).
    v256_ok: out (and res) rows 32-byte aligned with pitch % 16 == 0."""
    sms = sm_count() if sms is None else sms
    p = dict(cin=cin, cout=cout, taps=taps, sub=sub, up=up, fused2=kch2 > 0)
    NT = pick_nt(cout)
    if not (flags & 32) and NT % 32 == 0 and NT > 128:          # channel tiles of at most 128
        NT //= 2
    n_tiles = cout // NT
    Hp, Wp = H + 2, W + 2
    Qtot = N * Hp * Wp
    MT = min(2, max(1, 256 // NT))
    if MT == 2 and cdiv(Qtot, 512) * n_tiles < sms // 2:     # small problems: more, smaller items
        MT = 1
    halo = Wp + 1 if taps > 1 else 0
    need = 128 * MT + 2 * halo
    nseg = cdiv(need, 256)
    seg = (cdiv(need, nseg) + 7) & ~7
    P = seg * nseg
    a_chunk = (P * 32 + 255) & ~255
    b_chunk = taps * (NT // 2) * 32
    KCH = cin // 16
    KS = 1 if taps > 1 else min(KCH, 4)
    b2_chunk = (NT // 2) * 32
    budget = 212 * 1024
    pix_tiles = cdiv(Qtot, 256 * MT)
    items = pix_tiles * n_tiles
    pairs = max(1, min(sms // 2, items))
    b_res = 0
    if taps > 1 and not (flags & 64):
        bres_bytes = KCH * b_chunk + kch2 * b2_chunk
        pr = pairs - pairs % n_tiles                          # a pair keeps one channel tile
        if bres_bytes + 3 * a_chunk <= budget and pr >= n_tiles and items >= 3 * pr:
            b_res, pairs = 1, pr
    if b_res:
        stage = a_chunk
        S = min(12, (budget - KCH * b_chunk - kch2 * b2_chunk) // stage)
    else:
        stage = (KS * (a_chunk + b_chunk) + 1023) & ~1023
        S = min(12, budget // stage)
    v256 = bool(v256_ok) and not (flags & 128)
    p.update(NT=NT, n_tiles=n_tiles, Hp=Hp, Wp=Wp, Qtot=Qtot, MT=MT, nseg=nseg, seg=seg, P=P, KS=KS, b_res=b_res, S=S,
             pix_tiles=pix_tiles, items=items, pairs=pairs, grid=2 * pairs, v256=v256, vec_bias=bool(bias_aligned),
             vec_tbias=bool(tbias_vec), kernel=f"conv_tc2_kernel<{MT}, {9 if kch2 else taps}, {'true' if kch2 else 'false'}>")
    return p


def wg_pick_nt(cin):
    for nt in range(128, 15, -16):
        if cin % nt == 0:
            return nt
    return 0


def wg_plan(cin, cout, N, H, W, k, flags=0, sms=None):
    """wg_plan + wg_pair of conv_tc.cu (WG_KQ = 64 pixels per stage)."""
    sms = sm_count() if sms is None else sms
    NT = wg_pick_nt(cin)
    ntap = 3 if k == 3 else 1
    n_tiles, m_tiles = cin // NT, cdiv(cout, 128)
    Wp = W + 2
    Qtot = N * (H + 2) * Wp
    stages_total = cdiv(Qtot, 64)
    yz = ntap * n_tiles * m_tiles
    sp = sms // yz                                            # one wave: floor
    max_sp = max(1, (stages_total + 7) // 8)
    sp = max(1, min(sp, max_sp))
    spc = cdiv(stages_total, sp)
    splits = cdiv(stages_total, spc)
    pair = (not (flags & 1024)) and not (n_tiles > 2 and stages_total < 1500) and m_tiles % 2 == 0 and NT % 16 == 0
    ngrp = ntap * n_tiles
    ws = splits * m_tiles * ntap * n_tiles * 128 * ntap * NT * 4 + splits * ntap * n_tiles * m_tiles * 128 * 4
    grid = (m_tiles, ngrp, splits) if pair else (splits, ngrp, m_tiles)
    return dict(cin=cin, cout=cout, NT=NT, ntap=ntap, n_tiles=n_tiles, m_tiles=m_tiles, Qtot=Qtot, stages_total=stages_total,
                stages_per_cta=spc, splits=splits, pair=pair, ngrp=ngrp, workspace_bytes=ws, grid=grid,
                kernel="wgrad_tc2_kernel" if pair else "wgrad_tc_kernel")


def plan_str(p):
    keys = ("NT", "n_tiles", "MT", "nseg", "KS", "b_res", "S", "items", "pairs", "v256", "ntap", "m_tiles", "stages_total",
            "stages_per_cta", "splits", "pair", "kernel")
    return ", ".join(f"{k}={p[k]}" for k in keys if k in p)


# ================================================================================================================
# cases
# ================================================================================================================
def cv(name, N, cin, cout, H, W=None, k=3, op="fprop", bias=True, tbias=False, res=False, accum=False, c2=0,
       out_slice=None, flags=0):
    """Convolution case at kernel level: the kernel reads `cin` channels of an N x H x W input and writes `cout`.
    op 'dgrad' runs the flipped / transposed packed weight of a forward layer cout -> cin.  c2: channels of a fused 1x1
    second operand (a slice of a wider buffer).  out_slice: (c0, wide) -- out is channels [c0, c0 + cout) of a buffer with
    `wide` channels.  flags: ddpm_set_tc_mode path-forcing bits."""
    return dict(name=name, N=N, cin=cin, cout=cout, H=H, W=H if W is None else W, k=k, op=op, bias=bias, tbias=tbias,
                res=res, accum=accum, c2=c2, out_slice=out_slice, flags=flags)


def case_plan(c, sms=None):
    v256_ok = True
    if c["out_slice"] is not None:
        c0, wide = c["out_slice"]
        v256_ok = (2 * c0) % 32 == 0 and wide % 16 == 0
    return conv_plan(c["cin"], c["cout"], c["N"], c["H"], c["W"], c["k"] * c["k"], kch2=c["c2"] // 16, flags=c["flags"],
                     sms=sms, v256_ok=v256_ok)


B = 128                                                   # low-GPU UNet training batch
CONV_CASES = [
    # the low-GPU UNet's layers at their real batch
    cv("conv1 96->96@64 bias+tbias", B, 96, 96, 64, tbias=True),
    cv("dgrad 96->96@64", B, 96, 96, 64, op="dgrad", bias=False),
    cv("conv2 192->192@32 bias+res", B, 192, 192, 32, res=True),
    cv("dgrad 192->192@32", B, 192, 192, 32, op="dgrad", bias=False),
    cv("conv1 288->96@64", B, 288, 96, 64, tbias=True),
    cv("dgrad 96->288@64 (of 288->96)", B, 96, 288, 64, op="dgrad", bias=False),
    cv("conv1 384->192@32", B, 384, 192, 32, tbias=True),
    cv("conv1 384->192@16", B, 384, 192, 16, tbias=True),
    cv("conv 192->192@8", B, 192, 192, 8, tbias=True),
    cv("dgrad 192->192@8 accumulate", B, 192, 192, 8, op="dgrad", bias=False, accum=True),
    cv("skip 1x1 288->96@64", B, 288, 96, 64, k=1),
    cv("skip 1x1 384->192@32", B, 384, 192, 32, k=1),
    cv("skip 1x1 96->192@32", B, 96, 192, 32, k=1, res=True),
    cv("in conv 16->96@64", B, 16, 96, 64),
    cv("out conv 96->16@64", B, 96, 16, 64),
    cv("dgrad of out conv 16->96@64", B, 16, 96, 64, op="dgrad", bias=False),
    cv("conv2+skip 96 + 1x1 288 -> slice@64", B, 96, 96, 64, c2=288, out_slice=(0, 192)),
    cv("conv2+skip 192 + 1x1 384 -> slice@16", B, 192, 192, 16, c2=384, out_slice=(192, 384)),
    # CelebA256 layers (bench.py C256_SHAPES) at reduced batch, several items per CTA pair
    cv("c256 128->128@256", 2, 128, 128, 256, tbias=True),
    cv("c256 128->128@128", 4, 128, 128, 128, res=True),
    cv("c256 256->256@64", 8, 256, 256, 64),
    cv("c256 256->128@256", 2, 256, 128, 256),
    cv("c256 256->256@128", 2, 256, 256, 128),
    cv("c256 512->512@16", 64, 512, 512, 16, tbias=True),
    cv("c256 256->256@32", 16, 256, 256, 32),
    cv("c256 512->256@64", 4, 512, 256, 64),
    cv("c256 skip 1x1 384->128@128", 2, 384, 128, 128, k=1),
    # odd sizes, non-square images, tails, NT = 144, the remaining planner regimes
    cv("Cout 288 (NT 144) 96->288@16", 4, 96, 288, 16, res=True),
    cv("1x1 KS=2 32->96 odd", 3, 32, 96, 29, W=37, k=1),
    cv("1x1 KS=1 16->64 odd", 2, 16, 64, 21, W=19, k=1),
    cv("1x1 KS=4 MT=1 small 96->64", 1, 96, 64, 14, W=10, k=1),
    cv("items 73 96->96 nonsquare", 2, 96, 96, 92, W=97, tbias=True),
    cv("items 75 96->96 nonsquare", 2, 96, 96, 94, W=98),
    cv("small MT=1 192->192@8 N=2", 2, 192, 192, 8, res=True, accum=True),
    cv("tail MT=2 Qtot%512=1 96->96", 21, 96, 96, 41, W=53, res=True),
    cv("tail MT=2 Qtot%512=511 96->96", 19, 96, 96, 41, W=45),
    cv("tail MT=1 Qtot%256=1 96->96", 1, 96, 96, 17, W=25, res=True),
    cv("tail MT=1 Qtot%256=255 96->96", 1, 96, 96, 29, W=31),
    cv("tail Qtot%512 small 128->128", 7, 128, 128, 39, W=61),
    cv("items = machine pairs 96->96 48x45", 16, 96, 96, 48, W=45, tbias=True),
    cv("wide NT=192 (flag 32) 96->192@32", 8, 96, 192, 32, flags=32),
    cv("no b_res (flag 64) 192->192@32", 16, 192, 192, 32, flags=64, res=True),
    cv("128-bit epilogue (flag 128) 96->96@64", 8, 96, 96, 64, flags=128, res=True, accum=True, tbias=True),
    cv("128-bit epilogue: unaligned slice 96@32", 8, 96, 96, 32, out_slice=(8, 112), res=True),
]


def wg(name, N, cin, cout, H, W=None, k=3, bias=True, cin_valid=0, cout_valid=0, flags=0):
    return dict(name=name, N=N, cin=cin, cout=cout, H=H, W=H if W is None else W, k=k, bias=bias, cin_valid=cin_valid,
                cout_valid=cout_valid, flags=flags)


def wcase_plan(c, sms=None):
    return wg_plan(c["cin"], c["cout"], c["N"], c["H"], c["W"], c["k"], flags=c["flags"], sms=sms)


WGRAD_CASES = [
    wg("96->96@64", B, 96, 96, 64),
    wg("192->192@32 (pair)", B, 192, 192, 32),
    wg("192->192@32 single (flag 1024)", B, 192, 192, 32, flags=1024),
    wg("288->96@64", B, 288, 96, 64),
    wg("384->192@32 (pair)", B, 384, 192, 32),
    wg("384->192@16", B, 384, 192, 16),
    wg("192->192@8", B, 192, 192, 8),
    wg("1x1 288->96@64", B, 288, 96, 64, k=1),
    wg("1x1 384->192@32", B, 384, 192, 32, k=1),
    wg("in conv 16(3)->96@64", B, 16, 96, 64, cin_valid=3),
    wg("out conv 96->16(3)@64", B, 96, 16, 64, cout_valid=3),
    wg("c256 128->128@256", 2, 128, 128, 256),
    wg("c256 512->512@16 (m_tiles 4)", 16, 512, 512, 16),
    wg("c256 1x1 384->128@128", 2, 384, 128, 128, k=1),
    wg("m_tiles 3: 128->384 odd", 3, 128, 384, 29),
    wg("m_tiles 4 pair: 128->512@32", 8, 128, 512, 32),
    wg("NT 64: 64->128 nonsquare", 5, 64, 128, 30, W=41),
    wg("Cout 288 (m_tiles 3) 96->288@16", 4, 96, 288, 16),
    wg("pair odd tail 96->192", 3, 96, 192, 29),
]


# ================================================================================================================
# criteria (pure torch, any device)
# ================================================================================================================
def unit_stats(err, scale, unit, n_units):
    """Per unit: rms(err) and rms(scale)."""
    u = unit.reshape(-1)
    cnt = torch.bincount(u, minlength=n_units).double()
    e2 = torch.bincount(u, weights=err.reshape(-1).double() ** 2, minlength=n_units)
    s2 = torch.bincount(u, weights=scale.reshape(-1).double() ** 2, minlength=n_units)
    cnt = cnt.clamp(min=1)
    return (e2 / cnt).sqrt(), (s2 / cnt).sqrt()


def judge(got, ref, A, K, unit, n_units, bf16, extra_elem=None, extra_rms=None):
    """Criteria 1 and 2.  Returns (ok, c1, c2, worst_unit, detail): c1 = max |err| / per-element bound, c2 = max over
    units of rms(err) / unit bound (both must be <= 1).  extra_elem / extra_rms widen the bounds for an operand rounding
    the model does not contain (the summed phase weights of the folded up-sampling, the bf16 intermediate of up_bwd)."""
    got, ref, A = got.double(), ref.double(), A.double()
    err = got - ref
    E = K * U_ACC * A
    if extra_elem is not None:
        E = E + extra_elem
    bound = U_BF16 * (ref.abs() + E) + E if bf16 else E
    finite = bool(torch.isfinite(got).all())
    r1 = torch.where(bound > 0, err.abs() / bound, torch.where(err == 0, torch.zeros_like(err), torch.full_like(err, math.inf)))
    i1 = int(torch.argmax(r1)) if finite else 0
    c1 = float(r1.reshape(-1)[i1]) if finite else math.inf
    if bf16:
        rms_e, rms_r = unit_stats(err, ref, unit, n_units)
        ub = RMS_BF16 * rms_r
        if extra_rms is not None:
            _, rms_x = unit_stats(err, extra_rms, unit, n_units)
            ub = ub + U_BF16 * rms_x
    else:
        rms_e, rms_a = unit_stats(err, A, unit, n_units)
        ub = RMS_F32 * rms_a
    r2 = torch.where(ub > 0, rms_e / ub, torch.where(rms_e == 0, torch.zeros_like(rms_e), torch.full_like(rms_e, math.inf)))
    wu = int(torch.argmax(r2))
    c2 = float(r2[wu]) if finite else math.inf
    detail = dict(finite=finite, c1=c1, c2=c2, worst_elem=i1, worst_elem_got=float(got.reshape(-1)[i1]),
                  worst_elem_ref=float(ref.reshape(-1)[i1]), worst_unit=wu, worst_unit_rms_err=float(rms_e[wu]),
                  worst_unit_bound=float(ub[wu]))
    return finite and c1 <= 1.0 and c2 <= 1.0, c1, c2, wu, detail


def frobenius_1e2_accepts(got, ref):
    """The norm-relative check of test_gpu_tc.py / test_gpu_parity.py."""
    return float((got.double() - ref.double()).norm() / ref.double().norm()) < 1e-2


def bf16_round(t):
    return t.float().bfloat16().double() if t.dtype == torch.float64 else t.bfloat16().double()


# ================================================================================================================
# CPU tests: planner transcription, coverage, tolerances with teeth
# ================================================================================================================
def _wgrad_args_for(c):
    from ddpm_diffusion_model_b200 import _lib
    a = _lib.WgradArgs()
    a.act = _lib.Tensor(None, c["N"], c["H"], c["W"], c["cin"], c["cin"], 1)
    a.dy = _lib.Tensor(None, c["N"], c["H"], c["W"], c["cout"], c["cout"], 1)
    a.KH = a.KW = c["k"]
    a.stride, a.pad, a.dtype, a.prefer_tc = 1, c["k"] // 2, _lib.BF16, 1
    a.cin_valid, a.cout_valid = c["cin_valid"], c["cout_valid"]
    return _lib, a


def test_wgrad_plan_matches_library_workspace():
    """wg_plan reproduces the split-K partition the library sizes its workspace for (96->96@64, B = 128: 49 splits of
    178 stages, 21751296 bytes on a 148-SM device), for every weight-gradient case."""
    p = wg_plan(96, 96, 128, 64, 64, 3, sms=DEFAULT_SMS)
    assert (p["splits"], p["stages_per_cta"], p["workspace_bytes"]) == (49, 178, 21751296)
    for c in WGRAD_CASES:
        _lib, a = _wgrad_args_for(c)
        for fl in (0, 1024):              # the pair flag changes the kernel, not the workspace
            _lib.lib.ddpm_set_tc_mode(1 | (fl << 4), 0)
            try:
                got = int(_lib.lib.ddpm_wgrad_workspace_bytes(C.byref(a)))
            finally:
                _lib.lib.ddpm_set_tc_mode(1, 0)
            assert got == wcase_plan(c)["workspace_bytes"], (c["name"], got, wcase_plan(c))


def test_case_lists_reach_every_planner_regime():
    conv = [(c, case_plan(c)) for c in CONV_CASES]
    machine_pairs = sm_count() // 2
    need = {
        "MT 1": lambda c, p: p["MT"] == 1, "MT 2": lambda c, p: p["MT"] == 2,
        "nseg 1": lambda c, p: p["nseg"] == 1, "nseg > 1": lambda c, p: p["nseg"] > 1,
        "nseg >= 4 (W = 256)": lambda c, p: p["nseg"] >= 4,
        "KS 1 (1x1)": lambda c, p: p["taps"] == 1 and p["KS"] == 1, "KS 2": lambda c, p: p["KS"] == 2,
        "KS 4": lambda c, p: p["KS"] == 4,
        "b_res 0 (3x3)": lambda c, p: p["taps"] == 9 and p["b_res"] == 0, "b_res 1": lambda c, p: p["b_res"] == 1,
        "taps 9": lambda c, p: p["taps"] == 9, "taps 1": lambda c, p: p["taps"] == 1,
        "FUSED2": lambda c, p: p["fused2"], "FUSED2 + b_res": lambda c, p: p["fused2"] and p["b_res"],
        "dgrad": lambda c, p: c["op"] == "dgrad", "accumulate": lambda c, p: c["accum"],
        "residual": lambda c, p: c["res"], "time bias": lambda c, p: c["tbias"],
        "slice target": lambda c, p: c["out_slice"] is not None,
        "v256 0": lambda c, p: not p["v256"], "v256 0 unforced": lambda c, p: not p["v256"] and not (c["flags"] & 128),
        "NT 144": lambda c, p: p["NT"] == 144, "NT 192 (flag 32)": lambda c, p: p["NT"] == 192,
        "NT 16": lambda c, p: p["NT"] == 16,
        # items against the CTA pairs the machine holds: fewer (one item each), one fewer, one more (one pair walks two)
        "items < machine pairs": lambda c, p: p["items"] < machine_pairs,
        "items = machine pairs - 1": lambda c, p: p["items"] == machine_pairs - 1,
        "items = machine pairs + 1": lambda c, p: p["items"] == machine_pairs + 1,
        "items >= 3 x pairs, items % pairs != 0": lambda c, p: p["items"] >= 3 * p["pairs"] and p["items"] % p["pairs"],
        "Qtot % (256 MT) == 1": lambda c, p: p["Qtot"] % (256 * p["MT"]) == 1,
        "Qtot % (256 MT) small": lambda c, p: 2 <= p["Qtot"] % (256 * p["MT"]) <= 64,
        "Qtot % (256 MT) == 256 MT - 1": lambda c, p: p["Qtot"] % (256 * p["MT"]) == 256 * p["MT"] - 1,
        "non-square": lambda c, p: c["H"] != c["W"],
    }
    missing = [k for k, f in need.items() if not any(f(c, p) for c, p in conv)]
    # the compositions add: taps 4 (folded up-sampling), sub (stride 2), dgrad of the zero-interleaved stride-2 problem
    comp = [conv_plan(96, 96, 8, 32, 32, 4, up=True), conv_plan(96, 96, 16, 64, 64, 9, sub=True)]
    assert any(p["taps"] == 4 for p in comp) and any(p["sub"] for p in comp)
    assert not missing, missing
    wgp = [(c, wcase_plan(c)) for c in WGRAD_CASES]
    wneed = {
        "single": lambda c, p: not p["pair"], "pair": lambda c, p: p["pair"],
        **{f"m_tiles {m}": (lambda m: lambda c, p: p["m_tiles"] == m)(m) for m in (1, 2, 3, 4)},
        **{f"NT {nt}": (lambda nt: lambda c, p: p["NT"] == nt)(nt) for nt in (16, 64, 96, 128)},
        "stages_total % stages_per_cta != 0": lambda c, p: p["stages_total"] % p["stages_per_cta"] != 0,
        "Qtot % 64 != 0": lambda c, p: p["Qtot"] % 64 != 0,
        "cin_valid": lambda c, p: c["cin_valid"] > 0, "cout_valid": lambda c, p: c["cout_valid"] > 0,
        "bias, single, ngrp > 1": lambda c, p: c["bias"] and not p["pair"] and p["ngrp"] > 1,
        "bias, pair, ngrp > 1": lambda c, p: c["bias"] and p["pair"] and p["ngrp"] > 1,
        "1x1": lambda c, p: p["ntap"] == 1,
    }
    wmissing = [k for k, f in wneed.items() if not any(f(c, p) for c, p in wgp)]
    assert not wmissing, wmissing


def test_bf16_rounding_reaches_2_to_the_minus_8():
    """Why criterion 1 uses 2^-8 and not 2^-9: 1 + 2^-8 lies half-way between the bf16 neighbours 1 and 1 + 2^-7 and
    rounds (to even) to 1, an error of 2^-8 relative to the value."""
    v = torch.tensor([1.0 + 2.0 ** -8], dtype=torch.float64)
    r = bf16_round(v)
    assert float((r - v).abs() / v) > 2.0 ** -9
    assert float((r - v).abs() / v) <= 2.0 ** -8


def _block_case(seed=0, npix=128, nt=96, taps=9, cin=384):
    g = torch.Generator().manual_seed(seed)
    x = bf16_round(torch.randn(npix, taps, cin, generator=g, dtype=torch.float64))
    w = bf16_round(torch.randn(nt, taps, cin, generator=g, dtype=torch.float64) / math.sqrt(taps * cin))
    ref = torch.einsum("ptc,otc->po", x, w)
    A = torch.einsum("ptc,otc->po", x.abs(), w.abs())
    return x, w, ref, A


def test_teeth_a_missing_k_chunk_in_one_block():
    """(a) One 16-channel chunk of one tap missing from one 128-pixel block at K = 9 x 384."""
    x, w, ref, A = _block_case()
    K = 9 * 384
    unit = torch.zeros(ref.shape, dtype=torch.long)
    good = bf16_round(ref)
    assert judge(good, ref, A, K, unit, 1, True)[0]
    partial = torch.einsum("pc,oc->po", x[:, 4, 160:176], w[:, 4, 160:176])
    bad = bf16_round(ref - partial)
    ok, c1, c2, _, _ = judge(bad, ref, A, K, unit, 1, True)
    assert not ok and c2 > 4, (c1, c2)
    # the whole tensor: this block and 287 correct ones like it (the block repeated) -- the 1e-2 norm check passes it
    reps = 288
    whole_ref = ref.repeat(reps, 1)
    whole_bad = torch.cat([bad, good.repeat(reps - 1, 1)])
    assert frobenius_1e2_accepts(whole_bad, whole_ref)


def _stagewise_fp32(dy, x, spc):
    """Split-K like the kernel: fp32 sums of 64-pixel stages, fp32 accumulation over a split's stages, fp32 sum of the
    splits.  dy [K, co], x [K, ci] -> [co, ci], and the fp64 per-stage contributions [stages, co, ci]."""
    K = dy.shape[0]
    st = torch.einsum("skc,ski->sci", dy.reshape(K // 64, 64, -1), x.reshape(K // 64, 64, -1))
    st32 = st.float()
    splits = [st32[i:i + spc].sum(0) for i in range(0, st32.shape[0], spc)]
    tot = torch.zeros_like(splits[0])
    for s in splits:
        tot = tot + s
    return tot.double(), st


def test_teeth_b_dropped_and_doubled_stage_in_dw():
    """(b) dW over the reduction length of 96->96@64, B = 128 (524,288 pixels, 49 splits of 178 stages): one 64-pixel
    stage dropped, and one counted twice, in a (co tile, ci tile, tap) block of 4 x 4 channels."""
    g = torch.Generator().manual_seed(1)
    K = 128 * 64 * 64
    dy = bf16_round(torch.randn(K, 4, generator=g, dtype=torch.float64))
    x = bf16_round(torch.randn(K, 4, generator=g, dtype=torch.float64))
    ref = dy.t() @ x
    A = dy.abs().t() @ x.abs()
    good, st = _stagewise_fp32(dy, x, 178)
    unit = torch.zeros(ref.shape, dtype=torch.long)
    Kp = K + 49 + 1
    assert judge(good, ref, A, Kp, unit, 1, False)[0]
    for bad in (good - st[1234], good + st[5000]):
        ok, c1, c2, _, _ = judge(bad, ref, A, Kp, unit, 1, False)
        assert not ok and c2 > 2, (c1, c2)
    # the whole 3x3 gradient: this tap block and eight correct ones with the same statistics -- the 1e-2 norm check
    # passes the dropped stage
    assert frobenius_1e2_accepts(torch.cat([good - st[1234], good.repeat(8, 1)]), ref.repeat(9, 1))


def test_teeth_c_border_tap_missing_on_one_row():
    """(c) One border tap missing on a single image row: at row 17 of one image, the left-border pixel loses the tap
    (ky = 1, kx = 2) and the right-border pixel the tap (ky = 1, kx = 0) -- the taps that reach into the interior."""
    g = torch.Generator().manual_seed(2)
    N, Ci, Co, H, W = 2, 96, 32, 64, 64
    x = bf16_round(torch.randn(N, Ci, H, W, generator=g, dtype=torch.float64))
    w = bf16_round(torch.randn(Co, Ci, 3, 3, generator=g, dtype=torch.float64) / math.sqrt(9 * Ci))
    ref = F.conv2d(x, w, padding=1)
    A = F.conv2d(x.abs(), w.abs(), padding=1)
    good = bf16_round(ref)
    unit = conv_units(N, H, W, Co, Co, 1)
    n_units = int(unit.max()) + 1
    assert judge(good, ref, A, 9 * Ci, unit, n_units, True)[0]
    bad = good.clone()
    y = 17
    bad[1, :, y, 0] = bf16_round(ref[1, :, y, 0] - (w[:, :, 1, 2] * x[1, :, y, 1][None]).sum(1))
    bad[1, :, y, W - 1] = bf16_round(ref[1, :, y, W - 1] - (w[:, :, 1, 0] * x[1, :, y, W - 2][None]).sum(1))
    ok, c1, c2, _, _ = judge(bad, ref, A, 9 * Ci, unit, n_units, True)
    assert not ok and c1 > 1 and c2 > 1, (c1, c2)
    assert frobenius_1e2_accepts(bad, ref)


def test_teeth_d_bias_channel_short_by_one_stage():
    """(d) One channel of dbias short by one 64-pixel stage (524,288 pixels).  A lost stage of one channel is caught
    when its sum exceeds the 2^-18 rms(A) bound of the channel: for unit-variance dY that is the case for ~80 % of the
    stages; the stage used here is one of them, and the detection rate over every stage is asserted."""
    g = torch.Generator().manual_seed(3)
    K, Co = 128 * 64 * 64, 8
    dy = bf16_round(torch.randn(K, Co, generator=g, dtype=torch.float64))
    ref = dy.sum(0)
    A = dy.abs().sum(0)
    ones = torch.ones(K, 1, dtype=torch.float64)
    good, st = _stagewise_fp32(dy, ones, 178)
    good = good[:, 0]
    st = st[:, :, 0]
    unit = torch.arange(Co)
    Kp = K + 49 * 3 + 1
    assert judge(good, ref, A, Kp, unit, Co, False)[0]
    c = 5
    bound = RMS_F32 * float(A[c])
    stage = int(torch.argmax((st[:, c].abs() > 2 * bound).long()))       # the first stage with a clear sum
    bad = good.clone()
    bad[c] -= st[stage, c]
    ok, c1, c2, _, _ = judge(bad, ref, A, Kp, unit, Co, False)
    assert not ok and c2 > 1.5, (c1, c2)
    caught = float((st[:, c].abs() > bound + float((good[c] - ref[c]).abs())).double().mean())
    assert caught > 0.75, caught


# ================================================================================================================
# unit maps (which work unit produced each output element)
# ================================================================================================================
def conv_units(N, H, W, cout, NT, stride=1, device="cpu", up=False):
    """Unit id [N, cout, Ho, Wo] (NCHW like the reference) of every output element: (128-pixel block of the kernel's
    padded-linear Q, channel tile), and for the folded up-sampling also the phase.  H, W: the kernel input geometry."""
    Hp, Wp = H + 2, W + 2
    n_ct = cdiv(cout, NT)
    if up:
        Ho, Wo = 2 * H, 2 * W
        Y = torch.arange(Ho, device=device)
        X = torch.arange(Wo, device=device)
        yi, xi = Y // 2, X // 2
        ph = (Y % 2)[:, None] * 2 + (X % 2)[None, :]
    else:
        Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
        yi = torch.arange(Ho, device=device) * stride
        xi = torch.arange(Wo, device=device) * stride
        ph = torch.zeros(Ho, Wo, dtype=torch.long, device=device)
    n = torch.arange(N, device=device)
    q = (n[:, None, None] * Hp + yi[None, :, None] + 1) * Wp + xi[None, None, :] + 1       # [N, Ho, Wo]
    nblk = cdiv(N * Hp * Wp, 128)
    blk = ph[None] * nblk + q // 128
    co = torch.arange(cout, device=device) // NT
    return blk[:, None] * n_ct + co[None, :, None, None]


def wgrad_units(cout, cin, k, NT, device="cpu"):
    taps = k * k
    co = torch.arange(cout, device=device) // 128
    ci = torch.arange(cin, device=device) // NT
    t = torch.arange(taps, device=device)
    n_ci = cdiv(cin, NT)
    u = (co[:, None, None] * n_ci + ci[None, :, None]) * taps + t[None, None, :]
    return u.reshape(cout, cin, k, k)


# ================================================================================================================
# GPU helpers
# ================================================================================================================
def dev():
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def mods():
    from ddpm_diffusion_model_b200 import _lib, engine
    yield _lib, engine
    _lib.lib.ddpm_set_tc_mode(1, 0)
    _lib.lib.ddpm_set_force_simt(0)


def launched_kernels(fn):
    """Run fn under torch.profiler; [(name, grid)] of the CUDA kernels it launched."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            tr = json.load(f)
    out = []
    for e in tr.get("traceEvents", []):
        if e.get("cat") == "kernel":
            out.append((e.get("name", ""), tuple(e.get("args", {}).get("grid", ()))))
    return out


def with_mode(_lib, flags, fn):
    assert _lib.lib.ddpm_set_tc_mode(1 | (flags << 4), 0) == 0
    try:
        return fn()
    finally:
        _lib.lib.ddpm_set_tc_mode(1, 0)


def nchw64(a):
    return a.interior().double().permute(0, 3, 1, 2)


def report(kind, name, plan, c1, c2):
    # one line per case (run with -s): the margin of each criterion as a share of its bound
    print(f"\nMARGIN {kind} | {name} | c1 {c1:.3f} | c2 {c2:.3f} | {plan_str(plan)}")


def halo_zero(buf):
    t = buf
    return bool((t[:, 0] == 0).all() and (t[:, -1] == 0).all() and (t[:, :, 0] == 0).all() and (t[:, :, -1] == 0).all())


def spot_check_conv(x64, w64, ref, stride, pad, extra=None, n=256, seed=0):
    """Explicit CPU fp64 dot products for `n` random output elements of ref = conv2d(x64, w64) (+ extra)."""
    g = torch.Generator().manual_seed(seed)
    N, Co, Ho, Wo = ref.shape
    k = w64.shape[2]
    idx = [torch.randint(0, s, (n,), generator=g) for s in (N, Co, Ho, Wo)]
    xp = F.pad(x64, (pad, pad, pad, pad))
    worst = 0.0
    for i in range(n):
        nn_, co, yo, xo = (int(t[i]) for t in idx)
        patch = xp[nn_, :, yo * stride:yo * stride + k, xo * stride:xo * stride + k].cpu()
        v = float((patch * w64[co].cpu()).sum())
        if extra is not None:
            v += float(extra[nn_, co, yo, xo])
        r = float(ref[nn_, co, yo, xo])
        worst = max(worst, abs(v - r) / (abs(v) + 1e-300))
        assert abs(v - r) <= 1e-12 * (abs(v) + float((patch.abs() * w64[co].abs().cpu()).sum())), (i, v, r)
    return worst


def spot_check_wgrad(x64, dy64, ref, pad, n=32, seed=0):
    g = torch.Generator().manual_seed(seed)
    Co, Ci, k, _ = ref.shape
    N, _, H, W = dy64.shape
    xp = F.pad(x64, (pad, pad, pad, pad))
    for i in range(n):
        co, ci = int(torch.randint(0, Co, (1,), generator=g)), int(torch.randint(0, Ci, (1,), generator=g))
        ky, kx = int(torch.randint(0, k, (1,), generator=g)), int(torch.randint(0, k, (1,), generator=g))
        a = dy64[:, co].cpu()
        b = xp[:, ci, ky:ky + H, kx:kx + W].cpu()
        v = float((a * b).sum())
        s = float((a.abs() * b.abs()).sum())
        assert abs(v - float(ref[co, ci, ky, kx])) <= 1e-12 * (s + abs(v)), (co, ci, ky, kx)


# ================================================================================================================
# GPU: convolution
# ================================================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("case", CONV_CASES, ids=[c["name"] for c in CONV_CASES])
def test_conv_fp64(mods, case):
    _lib, engine = mods
    c = case
    torch.manual_seed(11)
    N, Ci, Co, H, W, k = c["N"], c["cin"], c["cout"], c["H"], c["W"], c["k"]
    dgrad = c["op"] == "dgrad"
    E = engine.Exec(dev(), _lib.BF16, False, False)
    # forward layer weight: [Co, Ci] for fprop; the data gradient runs the layer Ci <- Co, i.e. weight [Ci, Co]
    wshape = (Ci, Co, k, k) if dgrad else (Co, Ci, k, k)
    w = torch.nn.Parameter(torch.randn(*wshape, device=dev()) / math.sqrt(wshape[1] * k * k))
    wf, wd = E.wcache.get(E, w, _lib.BF16, dgrad)
    wb = w.detach().bfloat16()
    # the packed operand, bit for bit: fwd [Co][tap][Ci], dgrad [Ci_fwd][8 - tap][Co_fwd]
    if dgrad:
        wk = wb.flip(2, 3).transpose(0, 1).contiguous()          # [Co_kernel = fwd Cin, Ci_kernel = fwd Cout, k, k]
        assert torch.equal(wd.view(Co, k * k, Ci), wk.permute(0, 2, 3, 1).reshape(Co, k * k, Ci))
    else:
        wk = wb
        assert torch.equal(wf.view(Co, k * k, Ci), wk.permute(0, 2, 3, 1).reshape(Co, k * k, Ci))
    wpack = wd if dgrad else wf
    w64 = wk.double()

    x = E.act(N, H, W, Ci)
    x.interior().normal_()
    bias = torch.randn(Co, device=dev()) if c["bias"] else None
    tb = torch.randn(N, Co, device=dev()) if c["tbias"] else None
    res = None
    if c["res"]:
        res = E.act(N, H, W, Co)
        res.interior().normal_()
    in2 = w2pack = w2 = None
    if c["c2"]:
        wide_in = E.act(N, H, W, c["c2"] + 32)
        wide_in.interior().normal_()
        in2 = wide_in.slice(16, c["c2"])
        w2 = torch.nn.Parameter(torch.randn(Co, c["c2"], 1, 1, device=dev()) / math.sqrt(c["c2"]))
        w2pack, _ = E.wcache.get(E, w2, _lib.BF16, False)
    sentinel = 3.0
    if c["out_slice"] is not None:
        c0, wide = c["out_slice"]
        wide_out = E.act(N, H, W, wide)
        out = wide_out.slice(c0, Co)
    else:
        wide_out = E.act(N, H, W, Co)
        out = wide_out
    wide_out.interior().fill_(sentinel)
    if c["accum"]:
        out.interior().normal_()
    elif c["out_slice"] is None:
        out.interior().fill_(float("nan"))                       # an element the kernel forgets shows up
    acc0 = out.interior().double().permute(0, 3, 1, 2).clone() if c["accum"] else None
    before = wide_out.buf.t.clone()

    plan = case_plan(c)
    run = lambda: engine.conv(E, x, wpack, out, k, 1, k // 2, bias=bias, tbias=tb, res=res, accum=c["accum"],
                              in2=in2, w2pack=w2pack)
    ks = with_mode(_lib, c["flags"], lambda: launched_kernels(run))
    assert len(ks) == 1 and plan["kernel"] in ks[0][0], (ks, plan_str(plan))
    assert ks[0][1][0] == plan["grid"], (ks, plan_str(plan))

    # bit-exact side conditions
    after = wide_out.buf.t
    assert halo_zero(after), "the kernel wrote the zero halo"
    if c["out_slice"] is not None:
        c0, wide = c["out_slice"]
        keep = torch.ones(wide, dtype=torch.bool, device=dev())
        keep[c0:c0 + Co] = False
        assert torch.equal(after[..., keep], before[..., keep]), "channels outside the output slice changed"

    # fp64 reference and A
    x64 = nchw64(x)
    ref = F.conv2d(x64, w64, padding=k // 2)
    A = F.conv2d(x64.abs(), w64.abs(), padding=k // 2)
    K = k * k * Ci
    extra = torch.zeros_like(ref)
    if in2 is not None:
        x2 = nchw64(in2)
        w264 = w2.detach().bfloat16().double()
        extra = extra + F.conv2d(x2, w264)
        A += F.conv2d(x2.abs(), w264.abs())
        K += c["c2"]
    for t4 in ([bias.double()[None, :, None, None]] if bias is not None else []) + \
              ([tb.double()[:, :, None, None]] if tb is not None else []) + \
              ([nchw64(res)] if res is not None else []) + ([acc0] if acc0 is not None else []):
        extra = extra + t4
        A += t4.abs()
        K += 1
    spot_check_conv(x64, w64, ref, 1, k // 2)
    ref = ref + extra
    del extra
    got = nchw64(out)
    unit = conv_units(N, H, W, Co, plan["NT"], device=dev())
    n_units = int(unit.max()) + 1
    ok, c1, c2, wu, det = judge(got, ref, A, K, unit, n_units, True)
    report("conv", c["name"], plan, c1, c2)
    assert ok, (c["name"], plan_str(plan), det,
                f"worst unit {wu}: Q block {wu // plan['n_tiles']}, channel tile {wu % plan['n_tiles']}")


# ================================================================================================================
# GPU: weight gradient (+ bias gradient)
# ================================================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("case", WGRAD_CASES, ids=[c["name"] for c in WGRAD_CASES])
def test_wgrad_fp64(mods, case):
    _lib, engine = mods
    c = case
    torch.manual_seed(12)
    N, Ci, Co, H, W, k = c["N"], c["cin"], c["cout"], c["H"], c["W"], c["k"]
    E = engine.Exec(dev(), _lib.BF16, True, True)
    x = E.act(N, H, W, Ci)
    x.interior().normal_()
    dy = E.act(N, H, W, Co)
    dy.interior().normal_()
    ci_v = c["cin_valid"] or Ci
    co_v = c["cout_valid"] or Co
    w = torch.nn.Parameter(torch.zeros(co_v, ci_v, k, k, device=dev()))
    b = torch.nn.Parameter(torch.zeros(co_v, device=dev()))
    w.grad = torch.randn_like(w) * 0.1                           # the kernels accumulate into the gradient
    b.grad = torch.randn_like(b)
    g0, gb0 = w.grad.double().clone(), b.grad.double().clone()
    plan = wcase_plan(c)
    run = lambda: engine.wgrad(E, x, dy, w, k, 1, k // 2, bias=b if c["bias"] else None)
    ks = with_mode(_lib, c["flags"], lambda: launched_kernels(run))
    names = [n for n, _ in ks]
    assert len(ks) == 2 and plan["kernel"] + "(" in names[0] and "wgrad_reduce_kernel" in names[1], (names, plan_str(plan))
    assert ks[0][1] == plan["grid"], (ks, plan_str(plan))

    x64, dy64 = nchw64(x), nchw64(dy)
    ref = torch.nn.grad.conv2d_weight(x64, (Co, Ci, k, k), dy64, padding=k // 2)
    spot_check_wgrad(x64, dy64, ref, k // 2)
    A = torch.nn.grad.conv2d_weight(x64.abs(), (Co, Ci, k, k), dy64.abs(), padding=k // 2)[:co_v, :ci_v] + g0.abs()
    ref = ref[:co_v, :ci_v] + g0
    K = N * H * W + plan["splits"] + 1
    unit = wgrad_units(co_v, ci_v, k, plan["NT"], device=dev())
    ok, c1, c2, wu, det = judge(w.grad, ref, A, K, unit, int(unit.max()) + 1, False)
    report("wgrad", c["name"], plan, c1, c2)
    assert ok, (c["name"], plan_str(plan), det)
    if c["bias"]:
        refb = dy64.sum((0, 2, 3))[:co_v] + gb0
        Ab = dy64.abs().sum((0, 2, 3))[:co_v] + gb0.abs()
        Kb = N * H * W + plan["splits"] * plan["ngrp"] + 1
        ok, c1, c2, wu, det = judge(b.grad, refb, Ab, Kb, torch.arange(co_v, device=dev()), co_v, False)
        report("dbias", c["name"], plan, c1, c2)
        assert ok, (c["name"], "dbias", plan_str(plan), det)


# ================================================================================================================
# GPU: engine compositions, each against an fp64 reference of the module's own math
# ================================================================================================================
def _bf16_exact_(conv):
    with torch.no_grad():
        conv.weight.copy_(conv.weight.bfloat16().float())
        conv.bias.normal_()


@pytest.mark.gpu
def test_down_fwd_stride2_fp64(mods):
    _lib, engine = mods
    from ddpm_diffusion_model_b200.model.unet_backbone import Downsample
    torch.manual_seed(13)
    N, Cc, H = 64, 96, 64
    mod = Downsample(Cc).to(dev())
    E = engine.Exec(dev(), _lib.BF16, False, False)
    x = E.act(N, H, H, Cc)
    x.interior().normal_()
    plan = conv_plan(Cc, Cc, N, H, H, 9, sub=True)
    E.wcache.get(E, mod.conv.weight, _lib.BF16, False)           # pack and allocate outside the profiled region
    out = [E.act(N, H // 2, H // 2, Cc)]
    ks = launched_kernels(lambda: engine.down_fwd(E, mod, x, out[0]))
    assert len(ks) == 1 and plan["kernel"] in ks[0][0] and ks[0][1][0] == plan["grid"], (ks, plan_str(plan))
    y = out[0]
    assert halo_zero(y.buf.t)
    x64 = nchw64(x)
    w64 = mod.conv.weight.detach().bfloat16().double()
    b64 = mod.conv.bias.detach().double()
    ref = F.conv2d(x64, w64, b64, stride=2, padding=1)
    spot_check_conv(x64, w64, ref - b64[None, :, None, None], 2, 1)
    A = F.conv2d(x64.abs(), w64.abs(), b64.abs(), stride=2, padding=1)
    unit = conv_units(N, H, H, Cc, plan["NT"], stride=2, device=dev())
    ok, c1, c2, wu, det = judge(nchw64(y), ref, A, 9 * Cc + 1, unit, int(unit.max()) + 1, True)
    report("down_fwd", "96@64 stride 2", plan, c1, c2)
    assert ok, (plan_str(plan), det)


@pytest.mark.gpu
def test_down_bwd_zero_interleave_fp64(mods):
    """down_bwd on the tensor cores: dY is zero-interleaved to full resolution, then the stride-2 data gradient (accumulated
    into dx) and weight gradient run as stride-1 problems."""
    _lib, engine = mods
    from ddpm_diffusion_model_b200.model.unet_backbone import Downsample
    torch.manual_seed(14)
    N, Cc, H = 64, 96, 64
    mod = Downsample(Cc).to(dev())
    E = engine.Exec(dev(), _lib.BF16, True, True)
    x = E.act(N, H, H, Cc)
    x.interior().normal_()
    dout = E.act(N, H // 2, H // 2, Cc)
    dout.interior().normal_()
    dx = E.act(N, H, H, Cc)
    dx.interior().normal_()
    dx0 = nchw64(dx).clone()
    mod.conv.weight.grad = torch.randn_like(mod.conv.weight) * 0.1
    mod.conv.bias.grad = torch.randn_like(mod.conv.bias)
    g0, gb0 = mod.conv.weight.grad.double().clone(), mod.conv.bias.grad.double().clone()
    cplan = conv_plan(Cc, Cc, N, H, H, 9)
    wplan = wg_plan(Cc, Cc, N, H, H, 3)
    ks = launched_kernels(lambda: engine.down_bwd(E, mod, x, dout, dx, True))
    names = [n for n, _ in ks]
    assert any(cplan["kernel"] in n for n in names) and any(wplan["kernel"] + "(" in n for n in names), names
    torch.cuda.synchronize()
    assert halo_zero(dx.buf.t)
    x64, d64 = nchw64(x), nchw64(dout)
    w64 = mod.conv.weight.detach().bfloat16().double()
    ref = dx0 + F.conv_transpose2d(d64, w64, stride=2, padding=1, output_padding=1)
    A = dx0.abs() + F.conv_transpose2d(d64.abs(), w64.abs(), stride=2, padding=1, output_padding=1)
    unit = conv_units(N, H, H, Cc, cplan["NT"], device=dev())
    ok, c1, c2, wu, det = judge(nchw64(dx), ref, A, 9 * Cc + 1, unit, int(unit.max()) + 1, True)
    report("down_bwd dx", "96@64 zero-interleaved, accumulate", cplan, c1, c2)
    assert ok, (plan_str(cplan), det)
    refw = torch.nn.grad.conv2d_weight(x64, tuple(w64.shape), d64, stride=2, padding=1) + g0
    Aw = torch.nn.grad.conv2d_weight(x64.abs(), tuple(w64.shape), d64.abs(), stride=2, padding=1) + g0.abs()
    unit = wgrad_units(Cc, Cc, 3, wplan["NT"], device=dev())
    ok, c1, c2, wu, det = judge(mod.conv.weight.grad, refw, Aw, N * H * H + wplan["splits"] + 1, unit, int(unit.max()) + 1, False)
    report("down_bwd dW", "96@64 zero-interleaved", wplan, c1, c2)
    assert ok, (plan_str(wplan), det)
    refb = d64.sum((0, 2, 3)) + gb0
    Ab = d64.abs().sum((0, 2, 3)) + gb0.abs()
    ok, c1, c2, wu, det = judge(mod.conv.bias.grad, refb, Ab, N * H * H + wplan["splits"] * wplan["ngrp"] + 1,
                                torch.arange(Cc, device=dev()), Cc, False)
    report("down_bwd dbias", "96@64", wplan, c1, c2)
    assert ok, det


def _phase_weights64(w64):
    """fp64 [4][Co][Ci][2][2] phase weights of nearest-x2 + 3x3 (ddpm_pack_weights_up2x): S(0,0)={0}, S(0,1)={1,2},
    S(1,0)={0,1}, S(1,1)={2}."""
    S = {(0, 0): (0,), (0, 1): (1, 2), (1, 0): (0, 1), (1, 1): (2,)}
    Co, Ci = w64.shape[:2]
    pw = torch.zeros(4, Co, Ci, 2, 2, dtype=torch.float64, device=w64.device)
    for py in range(2):
        for px in range(2):
            for ty in range(2):
                for tx in range(2):
                    pw[2 * py + px, :, :, ty, tx] = sum(w64[:, :, ky, kx] for ky in S[(py, ty)] for kx in S[(px, tx)])
    return pw


@pytest.mark.gpu
def test_up_fwd_folded_phases_fp64(mods):
    """Sampling's up-sampling: four 2x2-tap phase convolutions of the low-resolution input (taps = 4) against fp64
    nearest-x2 + 3x3 built from the bf16 3x3 weights.  The parameter is made bf16-exact, so the only operand rounding
    beyond the model is the one rounding of each summed phase weight: |delta w| <= 2^-8 |sum w| (+ 3 * 2^-24 sum |w| for
    the fp32 sum), which adds 2^-8 * A_phase + 2^-22 * A per element and 2^-8 * rms(R), R^2 = sum x^2 (sum w)^2, per
    unit."""
    _lib, engine = mods
    from ddpm_diffusion_model_b200.model.unet_backbone import Upsample
    torch.manual_seed(15)
    N, Cc, H = 32, 192, 16
    mod = Upsample(Cc).to(dev())
    _bf16_exact_(mod.conv)
    E = engine.Exec(dev(), _lib.BF16, False, False)
    x = E.act(N, H, H, Cc)
    x.interior().normal_()
    plan = conv_plan(Cc, Cc, N, H, H, 4, up=True)
    E.wcache.get_up2x(E, mod.conv.weight, _lib.BF16)              # pack and allocate outside the profiled region
    out = [E.act(N, 2 * H, 2 * H, Cc)]
    ks = launched_kernels(lambda: engine.up_fwd(E, mod, x, out[0]))
    assert len(ks) == 4 and all(plan["kernel"] in n and g[0] == plan["grid"] for n, g in ks), (ks, plan_str(plan))
    y = out[0]
    assert halo_zero(y.buf.t)
    x64 = nchw64(x)
    w64 = mod.conv.weight.detach().double()
    b64 = mod.conv.bias.detach().double()
    pw = _phase_weights64(w64)
    wp = E.wcache.get_up2x(E, mod.conv.weight, _lib.BF16).double().view(4, Cc, 2, 2, Cc).permute(0, 1, 4, 2, 3)
    assert bool(((wp - pw).abs() <= U_BF16 * pw.abs() + 3 * 2.0 ** -24 * 4 * w64.abs().amax()).all())
    u64 = F.interpolate(x64, scale_factor=2, mode="nearest")
    ref = F.conv2d(u64, w64, b64, padding=1)
    spot_check_conv(u64, w64, ref - b64[None, :, None, None], 1, 1)
    A = F.conv2d(u64.abs(), w64.abs(), b64.abs(), padding=1)
    xp = F.pad(x64, (1, 1, 1, 1))
    A_ph = torch.zeros_like(ref)
    R = torch.zeros_like(ref)
    for ph in range(4):
        py, px = ph >> 1, ph & 1
        xs = xp[:, :, py:py + H + 1, px:px + H + 1]
        A_ph[:, :, py::2, px::2] = F.conv2d(xs.abs(), pw[ph].abs())
        R[:, :, py::2, px::2] = F.conv2d(xs * xs, pw[ph] * pw[ph]).sqrt()
    unit = conv_units(N, H, H, Cc, plan["NT"], device=dev(), up=True)
    ok, c1, c2, wu, det = judge(nchw64(y), ref, A, 4 * Cc + 1, unit, int(unit.max()) + 1, True,
                                extra_elem=U_BF16 * A_ph + U_ACC * A, extra_rms=R)
    report("up_fwd folded", "192@16 -> 32, 4 phases", plan, c1, c2)
    assert ok, (plan_str(plan), det)


@pytest.mark.gpu
def test_up_bwd_fp64(mods):
    """up_bwd: weight / bias gradient on the saved up-sampled input, the data gradient at full resolution (bf16), then
    the 2x2 sum to low resolution.  The bf16 intermediate du adds one rounding per summed term."""
    _lib, engine = mods
    from ddpm_diffusion_model_b200.model.unet_backbone import Upsample
    torch.manual_seed(16)
    N, Cc, H = 32, 192, 16
    mod = Upsample(Cc).to(dev())
    E = engine.Exec(dev(), _lib.BF16, True, True)
    x = E.act(N, H, H, Cc)
    x.interior().normal_()
    _, u = engine.up_fwd(E, mod, x)
    dout = E.act(N, 2 * H, 2 * H, Cc)
    dout.interior().normal_()
    mod.conv.weight.grad = torch.zeros_like(mod.conv.weight)
    mod.conv.bias.grad = torch.zeros_like(mod.conv.bias)
    cplan = conv_plan(Cc, Cc, N, 2 * H, 2 * H, 9)
    wplan = wg_plan(Cc, Cc, N, 2 * H, 2 * H, 3)
    out = [None]
    ks = launched_kernels(lambda: out.__setitem__(0, engine.up_bwd(E, mod, u, dout)))
    names = [n for n, _ in ks]
    assert any(cplan["kernel"] in n for n in names) and any(wplan["kernel"] + "(" in n for n in names), names
    dx = out[0]
    assert halo_zero(dx.buf.t)
    u64, d64 = nchw64(u), nchw64(dout)
    assert torch.equal(u64, F.interpolate(nchw64(x), scale_factor=2, mode="nearest"))
    w64 = mod.conv.weight.detach().bfloat16().double()
    du = F.conv_transpose2d(d64, w64, padding=1)
    Adu = F.conv_transpose2d(d64.abs(), w64.abs(), padding=1)
    Edu = 9 * Cc * U_ACC * Adu
    b_du = U_BF16 * (du.abs() + Edu) + Edu                       # per-element bound of each bf16 du term
    pool = lambda t: F.avg_pool2d(t, 2) * 4
    ref = pool(du)
    D = pool(b_du) + 3 * 2.0 ** -24 * pool(du.abs() + b_du)      # the four terms' bounds + their fp32 sum
    unit = conv_units(N, 2 * H, 2 * H, Cc, cplan["NT"], device=dev())[:, :, ::2, ::2]
    ok, c1, c2, wu, det = judge(nchw64(dx), ref, torch.zeros_like(ref), 0, unit, int(unit.max()) + 1, True,
                                extra_elem=D, extra_rms=pool(du * du).sqrt())
    report("up_bwd dx", "192@32 -> 16", cplan, c1, c2)
    assert ok, (plan_str(cplan), det)
    refw = torch.nn.grad.conv2d_weight(u64, tuple(w64.shape), d64, padding=1)
    Aw = torch.nn.grad.conv2d_weight(u64.abs(), tuple(w64.shape), d64.abs(), padding=1)
    unit = wgrad_units(Cc, Cc, 3, wplan["NT"], device=dev())
    ok, c1, c2, wu, det = judge(mod.conv.weight.grad, refw, Aw, N * 4 * H * H + wplan["splits"] + 1, unit,
                                int(unit.max()) + 1, False)
    report("up_bwd dW", "192@32", wplan, c1, c2)
    assert ok, (plan_str(wplan), det)
    ok, c1, c2, wu, det = judge(mod.conv.bias.grad, d64.sum((0, 2, 3)), d64.abs().sum((0, 2, 3)),
                                N * 4 * H * H + wplan["splits"] * wplan["ngrp"] + 1, torch.arange(Cc, device=dev()), Cc, False)
    report("up_bwd dbias", "192@32", wplan, c1, c2)
    assert ok, det
