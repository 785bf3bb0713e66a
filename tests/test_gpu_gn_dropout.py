"""GroupNorm + SiLU + dropout kernels against a float64 reference that rebuilds the dropout mask on the host.

The dropout mask is a counter hash (common.cuh): element e = ((n*H + y)*W + x)*C + c of the logical NHWC view,
wrapped to 32 bits, lies in word w = e >> 1 and is kept iff 16-bit half (e & 1) of lowbias32(((w & ~3) ^ key) + (w & 3))
>= thr16, with key = dropout_key(seed, step, layer).  The numpy emulator below is that definition; the CPU tests check the emulator
itself, the GPU tests check every kernel path against it:
  - bit for bit (gamma = 0, beta = 1: the output is exactly keep_scale or 0),
  - in float64 parity of the forward, the statistics and every backward variant,
  - with the forward and the backward on different paths (vector / scalar), which must draw the same mask,
  - across the dispatcher's envelope (cluster sizes, address paths, partial thread maps, ceilings),
  - for inputs with a large mean, and for a whole ResBlock called the way training calls it.

Tolerances (DESIGN §2, §4.2): fp32 element-wise |y - ref| <= 2e-5 max|ref| and norm-relative <= 3e-5; bf16 forward
per element 2^-8 |ref| + 2.5e-4 |z| keep_scale (tanh-SiLU) above an fp32 floor of 2e-5 max|ref|; bf16 gradients
norm-relative <= 2e-2 per tensor.
"""
import ctypes as C
import functools

import numpy as np
import pytest
import torch
import torch.nn.functional as F

M32 = 0xFFFFFFFF
U32 = np.uint32
DDPM_E_ARG = -1
EPS = 1e-6
SEEDS = (1234, (5 << 32) + 77)            # the second one exercises the seed >> 32 word of dropout_key
STEP = 1


# ------------------------------------------------------------------------------------------------
# host emulation of the mask (common.cuh: lowbias32, dropout_key, dropout_apply)
# ------------------------------------------------------------------------------------------------
def lowbias32(x):
    x = np.atleast_1d(np.asarray(x, dtype=np.uint32)).copy()
    with np.errstate(over="ignore"):
        x ^= x >> U32(16)
        x *= U32(0x7FEB352D)
        x ^= x >> U32(15)
        x *= U32(0x846CA68B)
        x ^= x >> U32(16)
    return x


def _lb(v):
    return int(lowbias32(v & M32)[0])


def dropout_key(seed, step, layer):
    k = _lb((seed & M32) ^ 0x9E3779B9)
    k = _lb(k ^ ((seed >> 32) & M32))
    k = _lb(k + (step & M32) * 0x85EBCA6B)
    return _lb(k ^ ((layer * 0xC2B2AE35) & M32))


def thr16(p):
    return int(np.float32(p) * np.float32(65536.0) + np.float32(0.5))


def keep_scale(p):
    return float(np.float32(1.0) / (np.float32(1.0) - np.float32(p)))


def hash_input(w, key):
    """The lowbias32 input of the uint32 word indices `w` (w = e >> 1)."""
    with np.errstate(over="ignore"):
        return ((w & ~U32(3)) ^ U32(key)) + (w & U32(3))


def keep_bits(e, key, thr):
    """Keep flags of the uint32 element indices `e`."""
    h = lowbias32(hash_input(e >> U32(1), key))
    half = np.where((e & U32(1)) != 0, h >> U32(16), h & U32(0xFFFF))
    return half >= thr


@functools.lru_cache(maxsize=8)
def keep_mask(N, H, W, Cc, key, thr):
    """bool [N, C, H, W]: the elements an N x H x W x C view keeps."""
    n = N * H * W * Cc
    assert n < 1 << 32
    e = np.arange(n, dtype=np.uint32)
    return torch.from_numpy(keep_bits(e, key, thr).reshape(N, H, W, Cc).transpose(0, 3, 1, 2).copy())


def layer_with_residue(seed, step, r):
    """The smallest layer id whose key has key & 3 == r (the hash input adds w & 3 to a block base whose low bits are
    key & 3, and the paths form that sum in different ways, so every low-bit pattern of the key has to occur)."""
    for layer in range(256):
        if dropout_key(seed, step, layer) & 3 == r:
            return layer
    raise AssertionError(f"no layer id < 256 with key & 3 == {r}")


# ------------------------------------------------------------------------------------------------
# CPU tests of the emulator
# ------------------------------------------------------------------------------------------------
def test_lowbias32_matches_the_scalar_definition():
    def ref(x):
        x ^= x >> 16; x = (x * 0x7FEB352D) & M32; x ^= x >> 15; x = (x * 0x846CA68B) & M32; x ^= x >> 16
        return x
    rs = np.random.RandomState(0)
    xs = np.concatenate([np.array([0, 1, 2, 0xFFFF, 0x10000, M32], dtype=np.uint32),
                         rs.randint(0, 1 << 32, size=1000, dtype=np.uint64).astype(np.uint32)])
    got = lowbias32(xs)
    assert [int(g) for g in got] == [ref(int(x)) for x in xs]
    assert int(lowbias32(0)[0]) == 0


def test_dropout_key_known_values():
    # key & 3 of seed 1234, step 1: layer 0 -> 1, layer 1 -> 0, layer 2 -> 3, layer 5 -> 3
    assert [dropout_key(1234, 1, layer) & 3 for layer in (0, 1, 2, 5)] == [1, 0, 3, 3]
    # every word of (seed, step, layer) reaches the key
    k = dropout_key(1234, 1, 3)
    assert len({k, dropout_key(1234 + (1 << 32), 1, 3), dropout_key(1235, 1, 3), dropout_key(1234, 2, 3),
                dropout_key(1234, 1, 4)}) == 5


def test_threshold_and_scale():
    assert thr16(0.1) == 6554 and thr16(0.5) == 32768 and thr16(0.25) == 16384
    assert keep_scale(0.5) == 2.0
    assert keep_scale(0.1) == float(np.float32(1) / np.float32(0.9))


@pytest.mark.parametrize("p", [0.1, 0.5])
def test_emulated_keep_rate(p):
    n = 1 << 20
    e = np.arange(n, dtype=np.uint32)
    want = 1.0 - thr16(p) / 65536.0
    sig = (want * (1 - want) / n) ** 0.5
    for key in (dropout_key(1234, 1, 1), dropout_key(SEEDS[1], 7, 2)):
        k = keep_bits(e, key, thr16(p))
        assert abs(k.mean() - want) < 5 * sig, (k.mean(), want)
        # per channel position of a bf16 packet (c mod 8 with C % 8 == 0) and per 16-bit half of the hash word
        for r in range(8):
            assert abs(k[r::8].mean() - want) < 5 * sig * 8 ** 0.5, (r, k[r::8].mean())
        for r in range(2):
            assert abs(k[r::2].mean() - want) < 5 * sig * 2 ** 0.5, (r, k[r::2].mean())


def test_emulated_mask_has_no_neighbour_correlation():
    n = 1 << 20
    for res in range(4):
        key = dropout_key(1234, STEP, layer_with_residue(1234, STEP, res))
        k = keep_bits(np.arange(n, dtype=np.uint32), key, thr16(0.5)).astype(np.float64)
        # lag 1: the two halves of one hash word; 2: adjacent words; 4, 6: across a block of four words;
        # 8: the same lane of the next bf16 packet
        for lag in (1, 2, 3, 4, 6, 8, 96):
            r = np.corrcoef(k[:-lag], k[lag:])[0, 1]
            assert abs(r) < 5 / n ** 0.5, (res, lag, r)


def test_hash_input_is_a_bijection_of_the_word_index():
    """No two words share a hash input (the + (w & 3) cannot carry into the next block), for every key & 3."""
    w = np.arange(1 << 20, dtype=np.uint32)
    for r in range(4):
        key = dropout_key(1234, STEP, layer_with_residue(1234, STEP, r))
        assert len(np.unique(hash_input(w, key))) == w.size, r
    # a bf16 packet (8 elements, e0 % 8 == 0) covers one block of four words: inputs (w0 ^ key) + i, i = 0..3 --
    # the one-XOR form the bf16 kernels use
    key = dropout_key(1234, STEP, layer_with_residue(1234, STEP, 3))
    w0 = np.arange(0, 1 << 16, 4, dtype=np.uint32)
    for i in range(4):
        with np.errstate(over="ignore"):
            assert np.array_equal(hash_input(w0 + U32(i), key), (w0 ^ U32(key)) + U32(i)), i
    # wraps at 2^32 like the kernels' uint32 arithmetic
    top = np.array([M32 - 3, M32 - 2, M32 - 1, M32], dtype=np.uint32)
    assert len(np.unique(hash_input(top, 0xFFFFFFFF))) == 4


def test_layer_ids_cover_every_key_residue():
    for seed in SEEDS:
        layers = [layer_with_residue(seed, STEP, r) for r in range(4)]
        assert [dropout_key(seed, STEP, L) & 3 for L in layers] == [0, 1, 2, 3]
        assert len(set(layers)) == 4


def test_mask_index_is_the_logical_nhwc_index():
    key, thr = dropout_key(1234, 1, 1), thr16(0.1)
    m = keep_mask(2, 3, 5, 16, key, thr)
    n, c, y, x = 1, 9, 2, 3
    e = np.array([((n * 3 + y) * 5 + x) * 16 + c], dtype=np.uint32)
    assert bool(m[n, c, y, x]) == bool(keep_bits(e, key, thr)[0])


# ------------------------------------------------------------------------------------------------
# GPU helpers
# ------------------------------------------------------------------------------------------------
TORCH_DT = {"f32": torch.float32, "bf16": torch.bfloat16}
SENTINEL = -3.25


def dev():
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def lib():
    from ddpm_diffusion_model_b200 import _lib, engine
    return _lib, engine


def _code(lib, dt):
    return lib[0].F32 if dt == "f32" else lib[0].BF16


def make_view(lib, dt, N, H, W, Cc, halo=1, offset=0, extra=0):
    """An NHWC view of Cc channels at channel `offset` of a buffer with Cc + extra channels per pixel.  The halo is
    zero; the channels outside the view hold a sentinel."""
    engine = lib[1]
    t = torch.zeros(N, H + 2 * halo, W + 2 * halo, Cc + extra, dtype=TORCH_DT[dt], device=dev())
    if extra:
        t[:, halo:halo + H, halo:halo + W, :offset] = SENTINEL
        t[:, halo:halo + H, halo:halo + W, offset + Cc:] = SENTINEL
    return engine.Act.wrap(t, N, H, W, Cc + extra, _code(lib, dt), halo).slice(offset, Cc)


LAYOUT = {"aligned": (1, 0, 0), "slice": (1, 8, 16), "halo0": (0, 0, 0), "misaligned": (1, 1, 3), "misaligned0": (0, 1, 2)}


def view(lib, dt, shape, layout="aligned"):
    N, Cc, H, W = shape
    halo, off, extra = LAYOUT[layout]
    return make_view(lib, dt, N, H, W, Cc, halo, off, extra)


def put(a, x):
    a.interior().copy_(x.permute(0, 2, 3, 1).to(a.buf.t.dtype))


def get(a):
    return a.interior().permute(0, 3, 1, 2).double()


def snap(a):
    return a.buf.t.clone()


def assert_outside_untouched(a, before, what=""):
    """Halo and the channels of the buffer outside the view are bitwise what they were."""
    t = a.buf.t
    h = a.halo
    out = torch.ones(t.shape, dtype=torch.bool, device=t.device)
    out[:, h:h + a.H, h:h + a.W, a.c0:a.c0 + a.C] = False
    iv = torch.int16 if t.dtype == torch.bfloat16 else torch.int32
    assert torch.equal(t.view(iv)[out], before.view(iv)[out]), f"{what}: a kernel wrote outside its view"


def stream():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def call_fwd(lib, kind, x, dt, G, stats, gamma, beta, act, p, rng, layer, out):
    fn = getattr(lib[0].lib, "ddpm_gn_fwd" if kind == "fwd" else "ddpm_gn_apply")
    return fn(C.byref(x.desc()), _code(lib, dt), G, stats.data_ptr(), gamma.data_ptr(), beta.data_ptr(), EPS, act, p,
              _p(rng) if p > 0 else None, layer, C.byref(out.desc()), stream())


def call_bwd(lib, variant, x, dt, G, stats, gamma, beta, act, p, rng, layer, dy, dx, accumulate, dgamma, dbeta,
             cs_nc=None, cs_c=None, scratch=0):
    L = lib[0].lib
    head = (C.byref(x.desc()), _code(lib, dt), G, stats.data_ptr(), gamma.data_ptr(), beta.data_ptr(), EPS, act, p,
            _p(rng) if p > 0 else None, layer, C.byref(dy.desc()), C.byref(dx.desc()), accumulate, _p(dgamma), _p(dbeta))
    if variant == "bwd":
        return L.ddpm_gn_bwd(*head, None, stream())
    return L.ddpm_gn_bwd_colsum(*head, _p(cs_nc), _p(cs_c), scratch, stream())


def group_sums(x, G):
    N = x.shape[0]
    xg = x.reshape(N, G, -1)
    return torch.stack([xg.sum(-1), (xg * xg).sum(-1)], -1)


def reference(x, gamma, beta, G, act, keep, scale, dy):
    """float64 GroupNorm -> SiLU -> mask * keep_scale and its gradients (autograd)."""
    xr = x.double().clone().requires_grad_(True)
    g = gamma.double().clone().requires_grad_(True)
    b = beta.double().clone().requires_grad_(True)
    z = F.group_norm(xr, G, g, b, EPS)
    y = F.silu(z) if act else z
    if keep is not None:
        y = y * keep.to(device=y.device, dtype=y.dtype) * scale
    y.backward(dy.double())
    return {"y": y.detach(), "z": z.detach(), "dx": xr.grad, "dgamma": g.grad, "dbeta": b.grad}


def check(name, got, ref, dt, fwd_z=None, scale=1.0, ref_scale=None):
    """AssertionError when `got` is outside the budget around the float64 `ref`.  `fwd_z`: the pre-activation of a bf16
    forward output (per-element bound).  `ref_scale`: magnitude to measure a near-cancelling sum against."""
    got, ref = got.double(), ref.double()
    d = (got - ref).abs()
    mx = float(ref.abs().max()) if ref_scale is None else float(ref_scale)
    nrel = float((got - ref).norm()) / max(float(ref.norm()), 1e-300)
    if ref_scale is not None:
        nrel = float((got - ref).norm()) / max(mx * ref.numel() ** 0.5, 1e-300)
    if dt == "f32":
        assert float(d.max()) <= 2e-5 * mx, f"{name}: max |err| {float(d.max()):.3e} > 2e-5 * {mx:.3e}"
        assert nrel <= 3e-5, f"{name}: norm-relative error {nrel:.3e} > 3e-5"
    elif fwd_z is not None:
        bound = 2.0 ** -8 * ref.abs() + 2.5e-4 * fwd_z.double().abs() * scale + 2e-5 * mx
        bad = d > bound
        assert not bool(bad.any()), f"{name}: {int(bad.sum())} of {bad.numel()} elements outside the bf16 bound " \
                                    f"(worst excess {float((d - bound).max()):.3e})"
    else:
        assert nrel <= 2e-2, f"{name}: norm-relative error {nrel:.3e} > 2e-2"
    return nrel


class Case:
    """Seeded inputs, parameters, mask and float64 reference of one GroupNorm(+SiLU)(+dropout) problem."""

    def __init__(self, dt, shape, G, act, p, layer=3, seed=SEEDS[0], mu=0.0, tseed=0, keep=None):
        N, Cc, H, W = shape
        self.dt, self.shape, self.G, self.act, self.p, self.layer = dt, shape, G, act, p, layer
        gen = torch.Generator(device=dev()).manual_seed(tseed)
        rnd = lambda *s: torch.randn(*s, generator=gen, device=dev(), dtype=torch.float64)  # noqa: E731
        self.x = (rnd(*shape) + mu).to(TORCH_DT[dt]).double()
        self.dy = rnd(*shape).to(TORCH_DT[dt]).double()
        self.gamma = (0.5 + torch.rand(Cc, generator=gen, device=dev(), dtype=torch.float64)).float()
        self.beta = rnd(Cc).float()
        self.rng = torch.tensor([seed, STEP], dtype=torch.int64, device=dev()) if p > 0 else None
        self.scale = keep_scale(p) if p > 0 else 1.0
        if keep is None and p > 0:
            keep = keep_mask(N, H, W, Cc, dropout_key(seed, STEP, layer), thr16(p)).to(dev())
        self.keep = keep
        self.ref = reference(self.x, self.gamma, self.beta, G, act, keep, self.scale, self.dy)
        self.ref_stats = group_sums(self.x, G)

    def with_keep(self, keep):
        c = object.__new__(Case)
        c.__dict__.update(self.__dict__)
        c.keep = keep
        c.ref = reference(self.x, self.gamma, self.beta, self.G, self.act, keep, self.scale, self.dy)
        return c

    def forward(self, lib, xl="aligned", ol="aligned", kind="fwd"):
        """Runs the forward; checks stats (fwd), the output and the untouched outside.  Returns the output view."""
        xv, ov = view(lib, self.dt, self.shape, xl), view(lib, self.dt, self.shape, ol)
        put(xv, self.x)
        before = snap(ov)
        if kind == "fwd":
            stats = torch.full((self.shape[0], self.G, 2), 1e30, dtype=torch.float64, device=dev())   # garbage
        else:
            stats = self.ref_stats.clone()
        rc = call_fwd(lib, kind, xv, self.dt, self.G, stats, self.gamma, self.beta, self.act, self.p, self.rng,
                      self.layer, ov)
        assert rc == 0, rc
        torch.cuda.synchronize()
        assert_outside_untouched(ov, before, f"{kind} out")
        if kind == "fwd":
            xa = self.x.reshape(self.shape[0], self.G, -1).abs()
            s, q = self.ref_stats[..., 0], self.ref_stats[..., 1]
            assert float(((stats[..., 0] - s).abs() / xa.sum(-1)).max()) < 1e-5, "stats: sum"
            assert float(((stats[..., 1] - q).abs() / q).max()) < 1e-5, "stats: sum of squares"
        return ov, stats

    def check_forward(self, ov, what="y"):
        return check(what, get(ov), self.ref["y"], self.dt, fwd_z=self.ref["z"], scale=self.scale)

    def backward(self, lib, stats, variant="colsum", scratch=0, accumulate=0, in_place=False, dyl="aligned",
                 dxl="aligned", xl="aligned"):
        """Runs one backward variant and checks dx, dgamma, dbeta and the column sums against the reference."""
        N, Cc, H, W = self.shape
        dt = self.dt
        xv = view(lib, dt, self.shape, xl)
        put(xv, self.x)
        dyv = view(lib, dt, self.shape, dyl)
        put(dyv, self.dy)
        gen = torch.Generator(device=dev()).manual_seed(99)
        base = None
        if in_place:
            dxv = dyv
            if accumulate:
                base = self.dy
        else:
            dxv = view(lib, dt, self.shape, dxl)
            if accumulate:
                base = (torch.randn(self.shape, generator=gen, device=dev(), dtype=torch.float64)
                        * float(self.ref["dx"].std())).to(TORCH_DT[dt]).double()
                put(dxv, base)
        dy_before, dx_before = snap(dyv), snap(dxv)
        g0 = torch.randn(Cc, generator=gen, device=dev())
        b0 = torch.randn(Cc, generator=gen, device=dev())
        dgamma, dbeta = g0.clone(), b0.clone()
        cs_nc = torch.full((N, Cc), 7.0, device=dev()) if variant == "colsum" else None
        c0 = torch.randn(Cc, generator=gen, device=dev())
        cs_c = c0.clone() if variant == "colsum" else None
        rc = call_bwd(lib, variant, xv, dt, self.G, stats, self.gamma, self.beta, self.act, self.p, self.rng, self.layer,
                      dyv, dxv, accumulate, dgamma, dbeta, cs_nc, cs_c, scratch)
        assert rc == 0, rc
        torch.cuda.synchronize()
        tag = f"{variant} scratch={scratch} acc={accumulate} in_place={in_place}"
        assert_outside_untouched(dxv, dx_before, tag + " dx")
        if not in_place:
            assert_outside_untouched(dyv, dy_before, tag + " dy")
            if not scratch:
                assert torch.equal(get(dyv), self.dy), tag + ": dy changed without dy_scratch"
        want = self.ref["dx"] if base is None else self.ref["dx"] + base
        got = get(dxv)
        check(tag + " dx", got, want, dt)
        check(tag + " dgamma", dgamma - g0, self.ref["dgamma"], dt)
        check(tag + " dbeta", dbeta - b0, self.ref["dbeta"], dt)
        if variant == "colsum":
            # channel sums of dx nearly cancel (GroupNorm gradients sum to zero per group): measure against sum |dx|
            check(tag + " colsum_nc", cs_nc, want.sum((2, 3)), dt, ref_scale=want.abs().sum((2, 3)).max())
            check(tag + " colsum_c", cs_c - c0, want.sum((0, 2, 3)), dt, ref_scale=want.abs().sum((0, 2, 3)).max())
            # and consistent with the dx the same launch wrote
            ctol = 1e-5 if dt == "f32" else 2e-3
            assert float((cs_nc - got.sum((2, 3))).abs().max()) <= ctol * float(got.abs().sum((2, 3)).max()), tag
        return got


def ids(v):
    return "x".join(map(str, v)) if isinstance(v, tuple) else str(v)


# ------------------------------------------------------------------------------------------------
# (b) the mask, bit for bit
# ------------------------------------------------------------------------------------------------
PATH_LAYOUTS = {"vector": ("aligned", "aligned"), "scalar_out": ("aligned", "misaligned"),
                "scalar_in": ("misaligned", "aligned")}


def _readout(lib, kind, dt, shape, G, p, seed, layer, xl, ol):
    """Output of the kernel with gamma = 0, beta = 1, act = none: exactly keep_scale where kept, 0 where dropped."""
    N, Cc, H, W = shape
    xv, ov = view(lib, dt, shape, xl), view(lib, dt, shape, ol)
    put(xv, torch.randn(shape, device=dev(), dtype=torch.float64))
    before = snap(ov)
    stats = group_sums(get(xv), G)
    gamma, beta = torch.zeros(Cc, device=dev()), torch.ones(Cc, device=dev())
    rng = torch.tensor([seed, STEP], dtype=torch.int64, device=dev())
    rc = call_fwd(lib, kind, xv, dt, G, stats, gamma, beta, 0, p, rng, layer, ov)
    assert rc == 0, rc
    torch.cuda.synchronize()
    assert_outside_untouched(ov, before, "readout")
    return get(ov)


def _assert_mask(y, keep, p, dt, what):
    bad = (y != 0) != keep
    assert not bool(bad.any()), f"{what}: {int(bad.sum())} of {bad.numel()} elements disagree with the documented mask"
    ks = torch.tensor(keep_scale(p), dtype=TORCH_DT[dt]).double().item()
    assert bool((y[keep] == ks).all()), f"{what}: kept elements are not exactly keep_scale"


@pytest.mark.gpu
@pytest.mark.parametrize("residue", [0, 1, 2, 3])
@pytest.mark.parametrize("path", list(PATH_LAYOUTS))
@pytest.mark.parametrize("dt", ["bf16", "f32"])
@pytest.mark.parametrize("kind", ["apply", "fwd"])
def test_mask_readout_is_bit_exact(lib, kind, dt, path, residue):
    shape, G = (2, 96, 6, 10), 32
    for seed in SEEDS:
        layer = layer_with_residue(seed, STEP, residue)
        for halo0 in (False, True):
            xl, ol = PATH_LAYOUTS[path]
            if halo0:
                xl, ol = ("misaligned0" if xl == "misaligned" else "halo0"), ("misaligned0" if ol == "misaligned" else "halo0")
            for p in (0.1, 0.5):
                y = _readout(lib, kind, dt, shape, G, p, seed, layer, xl, ol)
                keep = keep_mask(2, 6, 10, 96, dropout_key(seed, STEP, layer), thr16(p)).to(dev())
                _assert_mask(y, keep, p, dt, f"seed={seed} layer={layer} halo0={halo0} p={p}")


@pytest.mark.gpu
@pytest.mark.parametrize("dt", ["bf16", "f32"])
def test_mask_does_not_depend_on_layout(lib, dt):
    shape, G, p = (3, 64, 8, 12), 32, 0.1
    layer = layer_with_residue(SEEDS[0], STEP, 3)
    outs = [_readout(lib, "fwd", dt, shape, G, p, SEEDS[0], layer, "aligned", ol)
            for ol in ("aligned", "slice", "halo0", "misaligned")]
    for o in outs[1:]:
        assert torch.equal(o != 0, outs[0] != 0)


# ------------------------------------------------------------------------------------------------
# (c) float64 parity with dropout on, every backward variant
# ------------------------------------------------------------------------------------------------
BWD_VARIANTS = [("bwd", 0, 0, False), ("bwd", 0, 1, False)] + [
    ("colsum", s, a, ip) for s in (0, 1) for a in (0, 1) for ip in (False, True) if not (s and a and ip)]


@pytest.mark.gpu
@pytest.mark.parametrize("p", [0.0, 0.1, 0.5])
@pytest.mark.parametrize("act", [0, 1])
@pytest.mark.parametrize("dt", ["bf16", "f32"])
def test_parity_fp64_every_backward_variant(lib, dt, act, p):
    c = Case(dt, (3, 96, 12, 20), 32, act, p, layer=layer_with_residue(SEEDS[0], STEP, 3), tseed=7)
    ov, stats = c.forward(lib)
    c.check_forward(ov)
    for variant, scratch, acc, ip in BWD_VARIANTS:
        c.backward(lib, stats, variant, scratch, acc, ip)


# ------------------------------------------------------------------------------------------------
# (d) forward and backward on different paths
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("residue", [0, 1, 2, 3])
@pytest.mark.parametrize("pair", ["vector_fwd-scalar_bwd", "scalar_fwd-vector_bwd"])
@pytest.mark.parametrize("dt", ["bf16", "f32"])
def test_mixed_path_pair(lib, dt, pair, residue):
    c = Case(dt, (2, 96, 12, 12), 32, 1, 0.1, layer=layer_with_residue(SEEDS[0], STEP, residue), tseed=11)
    scalar_fwd = pair.startswith("scalar")
    ov, stats = c.forward(lib, ol="misaligned" if scalar_fwd else "aligned")
    c.check_forward(ov, "y (" + pair + ")")
    # the scalar backward comes from one misaligned tensor only: dx, then dy
    if scalar_fwd:
        c.backward(lib, stats, "colsum", 0, 0, False)
    else:
        c.backward(lib, stats, "colsum", 0, 0, False, dxl="misaligned")
        c.backward(lib, stats, "bwd", 0, 0, False, dyl="misaligned")


# ------------------------------------------------------------------------------------------------
# (e) the tolerances see a mask error
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("what", ["forward", "backward"])
def test_tolerances_catch_a_half_percent_mask_error(lib, what):
    c = Case("bf16", (4, 96, 32, 32), 32, 1, 0.1, layer=3, tseed=13)
    ov, stats = c.forward(lib)
    gen = torch.Generator(device=dev()).manual_seed(1)
    flip = torch.rand(c.keep.shape, generator=gen, device=dev()) < 0.005
    wrong = c.with_keep(c.keep ^ flip)
    if what == "forward":
        c.check_forward(ov)
        with pytest.raises(AssertionError):
            wrong.check_forward(ov)
    else:
        c.backward(lib, stats, "colsum", 1, 0, True)
        moved = float((wrong.ref["dx"] - c.ref["dx"]).norm() / c.ref["dx"].norm())
        assert moved > 0.04, moved                          # ~sqrt(0.005) = 7 % against a 2 % budget
        with pytest.raises(AssertionError):
            wrong.backward(lib, stats, "colsum", 1, 0, True)


# ------------------------------------------------------------------------------------------------
# (f) the dispatcher's envelope
# ------------------------------------------------------------------------------------------------
ENVELOPE = [
    # (dtype, (N, C, H, W), groups)
    ("bf16", (2, 32, 4, 4), 32),          # cluster 1; channels per group (1) < VEC
    ("f32", (2, 32, 8, 8), 32),           # the same for VEC 4
    ("bf16", (3, 96, 24, 24), 32),        # cluster 2; W = 24 is not a power of two (division address path)
    ("bf16", (2, 96, 12, 20), 32),        # W = 20, 12 channel vectors (256 % 12 != 0: inactive threads)
    ("bf16", (3, 96, 32, 32), 32),        # W = 32 (shift path)
    ("bf16", (2, 128, 32, 32), 32),       # cluster 4
    ("bf16", (4, 96, 64, 64), 32),        # cluster 8
    ("bf16", (2, 128, 128, 128), 32),     # cluster 16 (few large images)
    ("bf16", (2, 288, 16, 16), 32),       # 36 channel vectors
    ("f32", (2, 40, 16, 16), 8),          # 10 channel vectors of 4
    ("f32", (3, 96, 24, 24), 32),
    ("bf16", (2, 64, 16, 16), 8),         # 8 groups of 8 channels
    ("bf16", (130, 192, 16, 16), 32),     # many images
    ("bf16", (2, 2048, 4, 4), 32),        # the widest bf16 view (256 channel vectors)
    # the train step's norm2 shapes at B = 128
    ("bf16", (128, 96, 64, 64), 32),
    ("bf16", (128, 192, 32, 32), 32),
    ("bf16", (128, 192, 16, 16), 32),
    ("bf16", (128, 192, 8, 8), 32),
]


@pytest.mark.gpu
@pytest.mark.parametrize("dt,shape,G", ENVELOPE, ids=[f"{d}-{ids(s)}-G{g}" for d, s, g in ENVELOPE])
def test_envelope_train_step_path(lib, dt, shape, G):
    """bf16/fp32, p = 0.1, SiLU, the in-place scratch backward with column sums (what the UNet runs), all on channel
    slices of wider buffers whose other channels must stay untouched."""
    c = Case(dt, shape, G, 1, 0.1, layer=layer_with_residue(SEEDS[0], STEP, 3), tseed=shape[1])
    ov, stats = c.forward(lib, xl="slice", ol="slice")
    c.check_forward(ov)
    c.backward(lib, stats, "colsum", 1, 0, True, dyl="slice", xl="slice")


@pytest.mark.gpu
@pytest.mark.parametrize("dt,Cc,layout", [("bf16", 2056, "aligned"), ("bf16", 264, "misaligned"), ("f32", 264, "misaligned")])
def test_dispatch_ceiling_rejects_and_writes_nothing(lib, dt, Cc, layout):
    shape, G = (2, Cc, 4, 4), 8
    N = shape[0]
    xv, ov = view(lib, dt, shape, layout), view(lib, dt, shape, layout)
    dyv, dxv = view(lib, dt, shape, layout), view(lib, dt, shape, layout)
    for v in (xv, ov, dyv, dxv):
        v.buf.t.normal_()
    gamma, beta = torch.ones(Cc, device=dev()), torch.zeros(Cc, device=dev())
    rng = torch.tensor([SEEDS[0], STEP], dtype=torch.int64, device=dev())
    stats = torch.full((N, G, 2), 3.0, dtype=torch.float64, device=dev())
    dg, db = torch.full((Cc,), 5.0, device=dev()), torch.full((Cc,), 6.0, device=dev())
    cs_nc, cs_c = torch.full((N, Cc), 7.0, device=dev()), torch.full((Cc,), 8.0, device=dev())
    bufs = [ov.buf.t, dyv.buf.t, dxv.buf.t, stats, dg, db, cs_nc, cs_c]
    before = [b.clone() for b in bufs]
    for kind in ("fwd", "apply"):
        assert call_fwd(lib, kind, xv, dt, G, stats, gamma, beta, 1, 0.1, rng, 1, ov) == DDPM_E_ARG, kind
    rc = call_bwd(lib, "bwd", xv, dt, G, stats, gamma, beta, 1, 0.1, rng, 1, dyv, dxv, 0, dg, db)
    assert rc == DDPM_E_ARG
    for scratch in (0, 1):
        rc = call_bwd(lib, "colsum", xv, dt, G, stats, gamma, beta, 1, 0.1, rng, 1, dyv, dxv, 0, dg, db, cs_nc, cs_c, scratch)
        assert rc == DDPM_E_ARG
    torch.cuda.synchronize()
    for i, (a, b) in enumerate(zip(bufs, before)):
        assert torch.equal(a, b), f"buffer {i} written by a rejected call"


# ------------------------------------------------------------------------------------------------
# (g) inputs with a large mean
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dt,mu", [("f32", 0.0), ("f32", 8.0), ("bf16", 0.0), ("bf16", 8.0), ("bf16", 64.0)])
def test_large_mean_inputs(lib, dt, mu):
    """x = mu + N(0, 1): statistics sum x and x^2 in fp32 per thread and form E[x^2] - mu^2 in double; the backward
    subtracts mu * sum(dz) from sum(dz * x).  fp32 keeps its bound at mu/sigma = 8, bf16 its budget at 64."""
    c = Case(dt, (2, 64, 48, 48), 32, 1, 0.1, layer=1, mu=mu, tseed=17)
    ov, stats = c.forward(lib)
    c.check_forward(ov)
    c.backward(lib, stats, "colsum", 1, 0, True)
    c.backward(lib, stats, "bwd", 0, 0, False)


# ------------------------------------------------------------------------------------------------
# (h) a stand-alone ResBlock, called the way training calls it
# ------------------------------------------------------------------------------------------------
def _resblock_ref(blk, x, temb, dy, keep, scale):
    P = {k: v.detach().double().clone().requires_grad_(True) for k, v in blk.named_parameters()}
    xr = x.detach().double().clone().requires_grad_(True)
    tr = temb.detach().double().clone().requires_grad_(True)
    h = F.silu(F.group_norm(xr, blk.norm1.num_groups, P["norm1.weight"], P["norm1.bias"], blk.norm1.eps))
    h = F.conv2d(h, P["conv1.weight"], P["conv1.bias"], padding=1) + \
        F.linear(F.silu(tr), P["time_proj.1.weight"], P["time_proj.1.bias"])[:, :, None, None]
    h = F.silu(F.group_norm(h, blk.norm2.num_groups, P["norm2.weight"], P["norm2.bias"], blk.norm2.eps)) * keep * scale
    out = F.conv2d(h, P["conv2.weight"], P["conv2.bias"], padding=1)
    out = out + (F.conv2d(xr, P["skip.weight"], P["skip.bias"]) if "skip.weight" in P else xr)
    out.backward(dy.double())
    return out.detach(), xr.grad, tr.grad, {k: v.grad for k, v in P.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("cin,cout", [(64, 96), (96, 96)])
@pytest.mark.parametrize("dt", ["bf16", "f32"])
def test_resblock_with_dropout_matches_fp64(lib, dt, cin, cout):
    from ddpm_diffusion_model_b200 import functional as Fn
    from ddpm_diffusion_model_b200.model.unet_backbone import ResBlock
    torch.manual_seed(21)
    N, H, W, tdim, p = 4, 16, 16, 128, 0.1
    blk = ResBlock(cin, cout, tdim, dropout=p).to(dev()).train()
    with torch.no_grad():
        for m in (blk.norm1, blk.norm2):
            m.weight.uniform_(0.5, 1.5); m.bias.normal_()
    x = torch.randn(N, cin, H, W, device=dev())
    if dt == "bf16":
        x = x.bfloat16().float()
    x.requires_grad_(True)
    temb = torch.randn(N, tdim, device=dev(), requires_grad=True)
    dy = torch.randn(N, cout, H, W, device=dev())
    seed = SEEDS[1]
    Fn.seed_dropout(seed, dev())
    # the call advances the stream to step 1 and uses layer id 1 for norm2's dropout (functional.resblock_apply)
    if dt == "bf16":
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = blk(x, temb)
        dy = dy.bfloat16()
    else:
        out = blk(x, temb)
    out.backward(dy)
    torch.cuda.synchronize()
    keep = keep_mask(N, H, W, cout, dropout_key(seed, 1, 1), thr16(p)).to(dev()).double()
    ref_out, ref_dx, ref_dt, ref_g = _resblock_ref(blk, x, temb, dy, keep, keep_scale(p))
    if dt == "f32":
        check("out", out, ref_out, dt)
    else:
        assert float((out.double() - ref_out).norm() / ref_out.norm()) <= 2e-2   # after two bf16 convolutions
    check("dx", x.grad, ref_dx, dt)
    check("dtemb", temb.grad, ref_dt, dt)
    for k, prm in blk.named_parameters():
        check(k, prm.grad, ref_g[k], dt)
