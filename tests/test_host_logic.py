"""CPU-only tests: the C-ABI library loads and exports every declared symbol, the host-side mirror of
the reference interface (module tree, parameter order, schedules, drop-in aliases) is right, and the
data-parallel bucketing logic works over gloo with world_size 2.  No kernel is launched here."""
import ctypes
import json
import os
import re
import socket
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_abi_exports_every_declared_symbol():
    from ddpm_diffusion_model_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "ddpm_b200.h")).read()
    declared = set(re.findall(r"^\s*(?:int|int64_t)\s+(ddpm_\w+)\s*\(", hdr, flags=re.M))
    assert len(declared) >= 30
    lib = ctypes.CDLL(_lib.LIB_PATH)
    missing = [s for s in declared if not hasattr(lib, s)]
    assert not missing, missing
    # the ctypes table binds exactly the header's functions (+ the test hook ddpm_set_force_simt)
    assert declared <= set(_lib.SIGNATURES), declared - set(_lib.SIGNATURES)
    assert lib.ddpm_abi_version() == 2


def test_tc_mode_accepts_only_the_path_forcing_flags():
    """ddpm_set_tc_mode takes bit 0 = 1, base_offset 0 and flags 32 / 64 / 128 / 1024 in mode >> 4; it rejects anything
    else (such as the flags of removed experimental kernels) instead of silently ignoring it."""
    from ddpm_diffusion_model_b200 import _lib
    f = _lib.lib.ddpm_set_tc_mode
    try:
        for flags in (0, 32, 64, 128, 1024, 32 | 64 | 128 | 1024):
            assert f(1 | flags << 4, 0) == 0, flags
        for mode, base_offset in ((0, 0), (1, 1), (3, 0), (1 | 1 << 4, 0), (1 | 4 << 4, 0), (1 | 256 << 4, 0), (1 | 512 << 4, 0),
                                  (1 | 2048 << 4, 0), (1 | 4096 << 4, 0), (1 | (1024 | 2048) << 4, 0), (-1, 0)):
            assert f(mode, base_offset) == -1, (mode, base_offset)
    finally:
        assert f(1, 0) == 0


def test_struct_layouts_match_header():
    from ddpm_diffusion_model_b200 import _lib
    assert ctypes.sizeof(_lib.Tensor) == 32            # void* + 6 x int32
    assert ctypes.sizeof(_lib.AdamHyper) == 32
    assert _lib.ConvArgs.res.offset == _lib.ConvArgs.tbias_pitch.offset + 8   # padded to pointer alignment
    assert ctypes.sizeof(_lib.ConvArgs) % 8 == 0 and ctypes.sizeof(_lib.WgradArgs) % 8 == 0


def test_parameter_manifests_match_reference():
    from ddpm_diffusion_model_b200.model.unet_backbone import UNetDenoiser, build_unet_64x64
    man = json.load(open(os.path.join(ROOT, "tests", "golden", "param_manifests.json")))
    low = build_unet_64x64(base_channels=96, channel_mults=(1, 2, 2, 2), num_res_blocks=1, attn_resolutions={8},
                           num_heads=2, head_dim=32, dropout=0.1)
    big = UNetDenoiser(3, 128, (1, 1, 2, 2, 4), 2, {16}, 512, 0.1, 4, 64, 256)
    for name, m in (("low_gpu", low), ("celeba256", big), ("default64", build_unet_64x64())):
        assert [[k, list(p.shape)] for k, p in m.named_parameters()] == man[name], name
    assert sum(p.numel() for p in low.parameters()) == 12680259
    assert sum(p.numel() for p in big.parameters()) == 63100675


def test_state_dict_round_trip_with_reference_fixture(golden):
    from ddpm_diffusion_model_b200.model.unet_backbone import UNetDenoiser
    g = golden("unet_tiny_attn.pt")
    kw = dict(g["cfg"]); kw["attn_resolutions"] = set(kw["attn_resolutions"])
    m = UNetDenoiser(**kw)
    res = m.load_state_dict(g["state_dict"], strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    assert list(m.state_dict().keys()) == list(g["state_dict"].keys())


def test_diffusion_tables_and_api(golden):
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.model.difussion_utils import extract
    g = golden("tables.pt")
    for key, rec in g.items():
        d = Diffusion(**rec["kwargs"])
        assert list(d.state_dict().keys()) == []                      # non-persistent buffers
        for k, v in rec["tables"].items():
            assert torch.equal(getattr(d, k), v), (key, k)
    with pytest.raises(ValueError):
        Diffusion(schedule="nope")
    d = Diffusion()
    t = torch.tensor([-5, 3, 5000])
    out = extract(d.betas, t, torch.Size([3, 3, 8, 8]))
    assert out.shape == (3, 1, 1, 1) and t.tolist() == [0, 3, 999]     # in-place clamp, like the reference
    ts = d.sample_timesteps(4096)
    assert int(ts.min()) >= 1 and int(ts.max()) <= 999
    with pytest.raises(RuntimeError, match="CUDA-only"):
        d.q_sample(torch.zeros(1, 3, 4, 4), torch.zeros(1, dtype=torch.long))


def test_no_cpu_fallback_and_no_oracle_in_product():
    from ddpm_diffusion_model_b200.model.unet_backbone import build_unet_64x64
    m = build_unet_64x64(base_channels=32, channel_mults=(1, 2), num_res_blocks=1, attn_resolutions=set(), dropout=0.0)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(1, 3, 16, 16), torch.zeros(1, dtype=torch.long))
    pkg = os.path.join(ROOT, "ddpm-diffusion-model_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, f)).read()
                assert "import oracle" not in src and "from oracle" not in src and "/root/reference" not in src, f


def test_dropin_aliases():
    sys.path.insert(0, os.path.join(ROOT, "ddpm-diffusion-model_b200", "dropin"))
    try:
        for k in [k for k in sys.modules if k == "src" or k.startswith("src.")]:
            del sys.modules[k]
        from src.model.difussion_class import Diffusion                       # noqa: F401
        from src.model.unet_backbone import UNetDenoiser, ResBlock, Downsample, Upsample, build_unet_64x64  # noqa: F401
        from src.model.attention import SinusoidalPosEmb, TimeMLP, group_norm, AttnBlock   # noqa: F401
        from src.training_loops.train_one_epoch import train_one_epoch        # noqa: F401
        from src.training_loops.ema import EMA, ema_health, ema_reinit_from_model, ema_set_decay   # noqa: F401
        from src.training_loops.grad_scaler import make_grad_scaler, autocast_ctx   # noqa: F401
        from src.training_loops.training_utils import sample_ddpm, ddim_sample, compute_grad_norm   # noqa: F401
        from src.testing.ddpm_inference import ddpm_infer_sample, render_denoise_strip   # noqa: F401
        from src.testing.ddpim_inference import ddim_infer_sample, render_denoise_strip_ddim   # noqa: F401
        import inspect
        sig = inspect.signature(train_one_epoch)
        assert list(sig.parameters)[:4] == ["model", "diffusion", "dataloader", "optimizer"]
        assert sig.parameters["grad_clip"].default == 1.0 and sig.parameters["use_autocast"].default is True
        gn = group_norm(96)
        assert gn.num_groups == 32 and gn.eps == 1e-6
        assert make_grad_scaler("cuda", enabled=False) is None
    finally:
        sys.path.pop(0)


def test_ema_api_on_cpu_model():
    from ddpm_diffusion_model_b200.training_loops.ema import EMA, ema_health, ema_set_decay
    m = torch.nn.Linear(4, 4)
    e = EMA(m, decay=0.9)
    assert len(e.shadow) == 2 and torch.equal(e.shadow[0], m.weight)
    sd = e.state_dict()
    assert sd["decay"] == 0.9 and sd["shadow"] is e.shadow
    e2 = EMA(m, decay=0.5)
    e2.load_state_dict(sd)
    assert e2.decay == 0.9 and e2.shadow is sd["shadow"]
    ok, why, _ = ema_health(e, m)
    assert ok and why == "ok"
    ema_set_decay(e, 0.99)
    assert e.decay == 0.99
    with torch.no_grad():
        m.weight.add_(1.0)
    e.copy_to(m)
    assert torch.equal(m.weight, e.shadow[0])
    with pytest.raises(RuntimeError):
        e.update(m)                     # CPU parameters: no fallback


def test_ddim_schedules_match_oracle():
    from oracle import ddpm_oracle as O
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.testing.ddpim_inference import build_ddim_schedule
    from ddpm_diffusion_model_b200.training_loops.training_utils import ddim_timesteps
    d = Diffusion(T=1000)
    tb = O.make_tables()
    for steps in (2, 10, 50, 100, 1000):
        s = build_ddim_schedule(d, steps)
        assert s == O.ddim_schedule_t_linear(1000, steps)
        assert s[0] == 999 and s[-1] == 0 and all(a > b for a, b in zip(s, s[1:]))
    assert len(build_ddim_schedule(d, 50)) == 50                     # 49 transitions (SURVEY §3.2)
    assert build_ddim_schedule(d, 20, "alpha_bar_cosine") == O.ddim_schedule_alpha_bar(tb, 20)
    assert build_ddim_schedule(d, 5, schedule_idx=[10, 900, 400]) == [900, 400, 10, 0]
    with pytest.raises(ValueError):
        build_ddim_schedule(d, 5, "nope")
    for sch in ("linear", "cosine_alpha_bar", "karras"):
        assert ddim_timesteps(1000, 50, sch, "cpu").tolist() == O.ddim_sample_indices(1000, 50, sch).tolist()


def test_shard_range_partitions():
    from ddpm_diffusion_model_b200.dist import make_buckets, shard_range
    for n in (1, 7, 64, 513):
        for w in (1, 2, 4, 8):
            spans = [shard_range(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            assert max(h - l for l, h in spans) - min(h - l for l, h in spans) <= 1
    b = make_buckets(1000, 300)
    assert b == [(700, 1000), (400, 700), (100, 400), (0, 100)]
    # graded buckets: the start of the arena (the gradients that become final LAST) is cut into small pieces so that
    # only a small all-reduce is exposed in front of the optimiser pass
    b = make_buckets(1000, 300, tail_elems=250, tail_bucket_elems=100)
    assert b == [(700, 1000), (400, 700), (250, 400), (150, 250), (50, 150), (0, 50)]
    assert make_buckets(100, 300, tail_elems=5000, tail_bucket_elems=40) == [(60, 100), (20, 60), (0, 20)]


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _dp_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from ddpm_diffusion_model_b200.dist import GradSync, shard_range
        torch.manual_seed(0)
        n = 1000
        full = torch.randn(world, n)                     # every rank knows all ranks' gradients
        g = full[rank].clone()

        class M:                                         # stand-ins for sub-modules
            pass
        mods = [M() for _ in range(5)]
        spans = {id(m): (100 + 180 * i, 100 + 180 * (i + 1)) for i, m in enumerate(mods)}
        gs = GradSync(g, spans, bucket_bytes=4 * 256, tail_bytes=4 * 300, tail_bucket_bytes=4 * 64)
        assert len(gs.buckets) == 3 + 5 and gs.buckets[-1] == (0, 44)
        gs.begin()
        launched = []
        for m in reversed(mods):                         # backward order: highest offsets first
            gs.progress(m)
            launched.append(gs.next)
        assert launched == sorted(launched) and launched[0] >= 0 and gs.next < len(gs.buckets)
        gs.progress(None)                                # flush (time_mlp / in_conv region)
        assert gs.next == len(gs.buckets) and not gs.active
        ok = torch.allclose(g, full.mean(0), atol=1e-6)
        # a micro-batch that does not step must not communicate
        g2 = full[rank].clone()
        gs2 = GradSync(g2, spans, bucket_bytes=4 * 256, tail_bytes=0)
        gs2.reset()
        for m in reversed(mods):
            gs2.progress(m)
        ok = ok and torch.equal(g2, full[rank]) and shard_range(10) == ((0, 5) if rank == 0 else (5, 10))
        q.put((rank, bool(ok)))
    finally:
        dist.destroy_process_group()


def test_gradient_buckets_gloo_world2():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(30)
    assert res == [(0, True), (1, True)]


def test_checkpoint_format_is_the_reference_format(tmp_path, golden):
    """chekpoints.py:4-25: same dictionary; a file written here loads with plain torch.load (weights_only) and fits the
    reference's own load_ckpt: its model / optimiser / EMA entries line up, name for name and shape for shape, with the
    parameters of the reference's UNetDenoiser of the same configuration (recorded in golden/unet_tiny_attn.pt)."""
    from ddpm_diffusion_model_b200.model.unet_backbone import UNetDenoiser
    from ddpm_diffusion_model_b200.training_loops.chekpoints import load_ckpt, save_ckpt
    from ddpm_diffusion_model_b200.training_loops.ema import EMA
    kw = dict(in_channels=3, base_channels=32, channel_mults=(1, 2), num_res_blocks=1, attn_resolutions={8}, time_embed_dim=64,
              dropout=0.0, num_heads=2, head_dim=16, img_resolution=16)
    torch.manual_seed(0)
    model = UNetDenoiser(**kw)
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3)
    for p in model.parameters():                       # give the optimiser a state without running a kernel
        p.grad = torch.full_like(p, 1e-3)
    opt.step()
    ema = EMA(model, decay=0.99)
    scaler = torch.amp.GradScaler("cuda", enabled=False)
    path = str(tmp_path / "ck.pt")
    save_ckpt(path, model, opt, scaler, ema, step=7, extra={"epoch": 1, "global_step": 7})
    ck = torch.load(path, map_location="cpu", weights_only=True)
    assert set(ck) == {"model", "optimizer", "scaler", "ema", "step", "extra"}
    assert all(torch.equal(ck["model"][k], v) for k, v in model.state_dict().items())
    # no tensor drags a shared storage along
    assert ck["ema"]["shadow"][0].untyped_storage().nbytes() == ck["ema"]["shadow"][0].numel() * 4
    m2 = UNetDenoiser(**kw)
    o2 = torch.optim.AdamW(m2.parameters(), lr=1e-3)
    e2 = EMA(m2, decay=0.5)
    step, extra = load_ckpt(path, m2, o2, scaler, e2, map_location="cpu")
    assert step == 7 and extra == {"epoch": 1, "global_step": 7} and e2.decay == 0.99
    assert all(torch.equal(a, b) for a, b in zip(m2.state_dict().values(), model.state_dict().values()))
    assert torch.equal(o2.state[next(m2.parameters())]["exp_avg"], opt.state[next(model.parameters())]["exp_avg"])
    # what the reference's load_ckpt needs: a strict model.load_state_dict into its UNetDenoiser, optimizer.load_state_dict
    # for an AdamW over its parameters, and an EMA shadow per parameter
    g = golden("unet_tiny_attn.pt")
    assert {**g["cfg"], "attn_resolutions": set(g["cfg"]["attn_resolutions"])} == kw
    ref_sd, ref_names = g["state_dict"], g["param_names"]
    assert [(k, v.shape) for k, v in ck["model"].items()] == [(k, v.shape) for k, v in ref_sd.items()]
    ref_shapes = [ref_sd[k].shape for k in ref_names]
    assert [len(grp["params"]) for grp in ck["optimizer"]["param_groups"]] == [len(ref_names)]
    assert [ck["optimizer"]["state"][i]["exp_avg"].shape for i in range(len(ref_names))] == ref_shapes
    assert ck["ema"]["decay"] == 0.99 and [s.shape for s in ck["ema"]["shadow"]] == ref_shapes


def test_png_encoder_round_trips_through_pil():
    """Sampler output path (SURVEY 8(f) f3): the threaded PNG writer decodes to exactly the pixels it was given."""
    import io
    import numpy as np
    from PIL import Image
    from ddpm_diffusion_model_b200.testing._png import encode_png
    rng = np.random.default_rng(1)
    for shp in ((1, 1, 3), (7, 5, 3), (64, 64, 3), (130, 66, 3), (600, 300, 3), (33, 17, 1)):
        a = rng.integers(0, 256, shp, dtype=np.uint8)
        if shp[0] >= 64:
            a[: shp[0] // 2] = (np.arange(shp[1])[None, :, None] * 3 % 256).astype(np.uint8)      # compressible half
        for level in (0, 3, 9):
            im = np.asarray(Image.open(io.BytesIO(encode_png(a, level))))
            im = im[:, :, None] if shp[2] == 1 else im
            assert im.shape == a.shape and (im == a).all(), (shp, level)


def test_device_loader_epoch_order_matches_torch_dataloader():
    """Input side (SURVEY 8(f) f4): the feeder's permutation is drawn from the generator exactly like
    DataLoader(shuffle=True, generator=g) does, epoch after epoch."""
    from torch.utils.data import DataLoader, TensorDataset
    from ddpm_diffusion_model_b200.data.device_loader import DeviceLoader
    n = 53
    ref = DataLoader(TensorDataset(torch.arange(n)), batch_size=8, shuffle=True, generator=torch.Generator().manual_seed(21))
    g = torch.Generator().manual_seed(21)
    for _ in range(3):                                          # three complete epochs of the reference loader
        want = torch.cat([b[0] for b in ref])
        assert torch.equal(DeviceLoader.epoch_order(n, True, g), want)
    assert torch.equal(DeviceLoader.epoch_order(7, False, None), torch.arange(7))
    torch.manual_seed(9); a = DeviceLoader.epoch_order(n, True, None)
    torch.manual_seed(9); b = torch.cat([t[0] for t in DataLoader(TensorDataset(torch.arange(n)), batch_size=8, shuffle=True)])
    assert torch.equal(a, b)


def test_abi_struct_layouts_match_the_library():
    """The ctypes mirrors are checked against sizeof() inside the library at import; here field by field for the one
    struct whose tail grew this round (ddpm_conv_args: in2 / w2 appended, nothing before them moved)."""
    import ctypes as C
    from ddpm_diffusion_model_b200 import _lib
    got = (C.c_int32 * 6)()
    assert _lib.lib.ddpm_abi_struct_sizes(got, 6) == 6
    mine = [_lib.Tensor, _lib.ConvArgs, _lib.LinEntry, _lib.WgradArgs, _lib.PackEntry, _lib.AdamHyper]
    assert [int(v) for v in got] == [C.sizeof(t) for t in mine]
    assert _lib.ConvArgs.in2.offset + C.sizeof(_lib.Tensor) == _lib.ConvArgs.w2.offset and _lib.ConvArgs.bias_n.offset < _lib.ConvArgs.in2.offset


def test_device_loader_shards_partition_the_epoch():
    """Under data parallelism every rank walks a disjoint, equally sized share of the SAME permutation."""
    from ddpm_diffusion_model_b200.data.device_loader import DeviceLoader
    n, world = 103, 4
    order = DeviceLoader.epoch_order(n, True, torch.Generator().manual_seed(3))
    parts = [DeviceLoader.shard_order(order, r, world) for r in range(world)]
    assert all(p.numel() == n // world for p in parts)
    merged = torch.stack(parts, 1).reshape(-1)                    # interleave back
    assert torch.equal(merged, order[:(n // world) * world])
    assert torch.equal(DeviceLoader.shard_order(order, 0, 1), order)


# ------------------------------------------------------------------------------------------------
# baseline arms: the unmodified reference, vendored; the reference process maps no product code
# ------------------------------------------------------------------------------------------------
def test_vendored_reference_is_byte_identical_and_untracked():
    import hashlib
    import json
    import subprocess
    ref = "/root/reference/src"
    man = os.path.join(ROOT, "baseline", "_ref", "MANIFEST.json")
    if not os.path.isdir(ref):
        if not os.path.exists(man):
            pytest.skip("no /root/reference and no vendored copy")
    else:
        subprocess.check_call([sys.executable, os.path.join(ROOT, "tools", "vendor_reference.py")])
    files = json.load(open(man))["files"]
    assert len(files) >= 16 and "src/training_loops/train_one_epoch.py" in files
    for rel_path, sha in files.items():
        got = hashlib.sha256(open(os.path.join(ROOT, "baseline", "_ref", rel_path), "rb").read()).hexdigest()
        assert got == sha, rel_path
        if os.path.isdir(ref):
            assert hashlib.sha256(open(os.path.join("/root/reference", rel_path), "rb").read()).hexdigest() == sha
    tracked = subprocess.run(["git", "-C", ROOT, "ls-files", "baseline/_ref"], capture_output=True, text=True).stdout.strip()
    assert tracked == "", "baseline/_ref must stay out of the history"


def test_reference_arm_runs_the_reference_and_never_imports_the_product():
    """`bench.py --impl reference` (tiny bounded sample): the line says kind=reference, and the process that produced it
    has neither the product package nor the oracle nor libddpm_b200.so mapped."""
    import json
    import subprocess
    if not os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "src")):
        pytest.skip("reference not vendored")
    code = (
        "import sys, json, runpy, os\n"
        f"sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', '--warmup', '0', '--ref-quick', '--ref-batch', '2']\n"
        f"runpy.run_path({os.path.join(ROOT, 'bench.py')!r}, run_name='__main__')\n"
        "bad = [m for m in sys.modules if m.startswith('ddpm_diffusion_model_b200') or m.startswith('oracle')]\n"
        "maps = open('/proc/self/maps').read()\n"
        "sys.stderr.write('CHECK ' + json.dumps({'bad': bad, 'so': 'libddpm_b200' in maps}) + '\\n')\n"
    )
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["impl"] == "reference" and line["cpu_baseline"]["kind"] == "reference" and line["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["config"]["reference_tree"] != "unknown"
    chk = json.loads([ln for ln in out.stderr.splitlines() if ln.startswith("CHECK ")][-1][6:])
    assert chk == {"bad": [], "so": False}, chk


def test_graph_step_is_only_used_for_pure_steps():
    """train_one_epoch replays a captured CUDA graph only when the step has no host-side effects a replay would skip:
    this package's own Diffusion / UNetDenoiser methods, no instance-level overrides, no hooks (host logic, no GPU needed)."""
    import torch
    from ddpm_diffusion_model_b200.model.difussion_class import Diffusion
    from ddpm_diffusion_model_b200.model.unet_backbone import UNetDenoiser
    from ddpm_diffusion_model_b200.training_loops.train_one_epoch import _pure_step

    model = UNetDenoiser(3, 32, (1, 2), 1, {8}, 64, 0.0, 2, 16, 16)
    diff = Diffusion(T=10, img_size=16)
    assert _pure_step(model, diff)
    # a test / user that feeds its own timesteps or noise through an instance attribute: every step must run eagerly
    diff.sample_timesteps = lambda B, device=None: torch.zeros(B, dtype=torch.long)
    assert not _pure_step(model, diff)
    del diff.sample_timesteps
    assert _pure_step(model, diff)
    h = model.in_conv.register_forward_hook(lambda m, i, o: None)
    assert not _pure_step(model, diff)
    h.remove()
    assert _pure_step(model, diff)
    model.forward = lambda x, t: x
    assert not _pure_step(model, diff)
    del model.forward

    class Sub(UNetDenoiser):
        pass
    assert not _pure_step(Sub(3, 32, (1, 2), 1, {8}, 64, 0.0, 2, 16, 16), diff)
