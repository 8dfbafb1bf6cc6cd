"""CPU tests (-m "not gpu"): the C-ABI library loads and exports every symbol include/ladi_b200.h declares (no compute calls
without a GPU), weight packing matches the kernel's K-segment walk, host-side pipeline validation, the no-CPU-fallback rule,
and the N>1 sharding logic over a world_size-2 gloo group."""
import os
import re
import subprocess

import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from ladi_vton_b200 import lib
    hdr = open(os.path.join(ROOT, "include", "ladi_b200.h")).read()
    declared = set(re.findall(r"LADI_API\s+[\w\s\*]+?\b(ladi_\w+)\s*\(", hdr))
    assert len(declared) >= 19
    assert declared == set(lib.SIGNATURES), declared ^ set(lib.SIGNATURES)
    l = lib.load()  # raises if the .so is missing; getattr raises on a missing export
    for name in declared:
        assert hasattr(l, name)
    assert l.ladi_abi_version() == lib.ABI_VERSION == 2
    out = subprocess.run(["nm", "-D", "--defined-only", lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (ladi_\w+)", out))
    assert declared <= exported


def test_no_cpu_fallback():
    """Without a CUDA device the product path must fail loudly, never fall back to the oracle or to PyTorch ops."""
    import ladi_vton_b200 as L
    from ladi_vton_b200 import ops, weights
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    with pytest.raises(RuntimeError):
        ops.gemm(torch.zeros(8, 64, dtype=torch.bfloat16), weights.pack_linear(torch.zeros(8, 64)), 8)
    with pytest.raises(RuntimeError, match="CUDA"):
        L.UNet2DConditionModel().to("cpu")
    src = "".join(open(os.path.join(ROOT, "ladi_vton_b200", f)).read() for f in os.listdir(os.path.join(ROOT, "ladi_vton_b200")) if f.endswith(".py"))
    assert "ladi_oracle" not in src and "import oracle" not in src  # the product never imports the checker


def _emulated_conv(xs, packed, sc=None, stride=1, pad_lo=1, ksize=3):
    """CPU restatement of ladi_conv2d_bf16's K-segment walk (taps row-major x sources, 64-channel blocks with zero fill,
    then the 1x1 shortcut segments) -- checks weights.pack_conv against F.conv2d."""
    n, _, h, w = xs[0].shape
    ho, wo = ((h + (2 if pad_lo else 1) - 3) // 2 + 1, (w + (2 if pad_lo else 1) - 3) // 2 + 1) if stride == 2 else (h, w)
    cols = []
    for ky in range(ksize):
        for kx in range(ksize):
            for x in xs:
                c = x.shape[1]
                cp = (c + 63) // 64 * 64
                xp = F.pad(x, (2, 2, 2, 2))
                oy, ox = (ky - pad_lo, kx - pad_lo) if ksize == 3 else (0, 0)
                patch = xp[:, :, 2 + oy: 2 + oy + (ho - 1) * stride + 1: stride, 2 + ox: 2 + ox + (wo - 1) * stride + 1: stride]
                cols.append(F.pad(patch, (0, 0, 0, 0, 0, cp - c)))
    for x in sc or []:
        c = x.shape[1]
        cols.append(F.pad(x, (0, 0, 0, 0, 0, (c + 63) // 64 * 64 - c)))
    a = torch.cat(cols, dim=1).permute(0, 2, 3, 1).reshape(n * ho * wo, -1)
    assert a.shape[1] == packed.shape[1]
    return (a @ packed.float().t()).reshape(n, ho, wo, -1).permute(0, 3, 1, 2)


@pytest.mark.parametrize("cs,stride,pad_lo", [([64], 1, 1), ([31], 1, 1), ([128, 64], 1, 1), ([96], 2, 1), ([64], 2, 0)])
def test_pack_conv_matches_kernel_k_walk(cs, stride, pad_lo):
    from ladi_vton_b200 import weights
    g = torch.Generator().manual_seed(0)
    xs = [torch.randn(2, c, 8, 6, generator=g) for c in cs]
    w = torch.randn(40, sum(cs), 3, 3, generator=g)
    packed = weights.pack_conv(w, cs).float()
    x = torch.cat(xs, 1)
    ref = F.conv2d(F.pad(x, (0, 1, 0, 1)) if (stride == 2 and pad_lo == 0) else x, w.bfloat16().float(), stride=stride,
                   padding=0 if (stride == 2 and pad_lo == 0) else 1)
    got = _emulated_conv(xs, packed, stride=stride, pad_lo=pad_lo)
    assert got.shape == ref.shape
    assert torch.allclose(got, ref, atol=1e-3, rtol=1e-3)


def test_pack_conv_shortcut_and_geglu_and_linear():
    from ladi_vton_b200 import weights
    g = torch.Generator().manual_seed(1)
    hmid, x0, x1 = torch.randn(1, 64, 4, 4, generator=g), torch.randn(1, 96, 4, 4, generator=g), torch.randn(1, 32, 4, 4, generator=g)
    w, ws = torch.randn(24, 64, 3, 3, generator=g), torch.randn(24, 128, 1, 1, generator=g)
    packed = weights.pack_conv(w, [64], ws, [96, 32])
    assert packed.shape == (24, 9 * 64 + 128 + 64)
    ref = F.conv2d(hmid, w.bfloat16().float(), padding=1) + F.conv2d(torch.cat([x0, x1], 1), ws.bfloat16().float())
    assert torch.allclose(_emulated_conv([hmid], packed, sc=[x0, x1]), ref, atol=1e-3, rtol=1e-3)
    wi, bi = weights.interleave_geglu(torch.arange(8.0)[:, None].repeat(1, 3), torch.arange(8.0))
    assert bi.tolist() == [0, 4, 1, 5, 2, 6, 3, 7] and wi[:, 0].tolist() == bi.tolist()
    assert weights.pack_linear(torch.ones(5, 70)).shape == (5, 128)


def test_pack_conv_up2x_matches_upsample_then_conv():
    """weights.pack_conv_up2x (sub-pixel form of diffusers Upsample2D: nearest-2x + conv3x3) walked like ladi_conv2d_bf16's up2x mode does --
    per output parity (py, px): 4 taps (ty, tx) reading input pixel (i + py - 1 + ty, j + px - 1 + tx), K order = taps row-major x 64-channel blocks,
    weight rows [parity * c_out, (parity + 1) * c_out) -- against F.conv2d(F.interpolate(x, 2, 'nearest'))."""
    from ladi_vton_b200 import weights
    g = torch.Generator().manual_seed(2)
    ci, co, h, w = 96, 40, 6, 5
    x = torch.randn(2, ci, h, w, generator=g)
    wt = torch.randn(co, ci, 3, 3, generator=g)
    packed = weights.pack_conv_up2x(wt, [ci]).float()
    cp = (ci + 63) // 64 * 64
    assert packed.shape == (4 * co, 4 * cp)
    ref = F.conv2d(F.interpolate(x, scale_factor=2, mode="nearest"), wt, padding=1)
    out = torch.zeros_like(ref)
    xp = F.pad(x, (1, 1, 1, 1, 0, cp - ci))  # zero padding = TMA out-of-bounds fill; channel padding = zero weights
    for par in range(4):
        py, px = par >> 1, par & 1
        cols = [xp[:, :, py + ty: py + ty + h, px + tx: px + tx + w] for ty in (0, 1) for tx in (0, 1)]
        a = torch.cat(cols, dim=1).permute(0, 2, 3, 1).reshape(-1, 4 * cp)
        y = (a @ packed[par * co:(par + 1) * co].t()).reshape(2, h, w, co).permute(0, 3, 1, 2)
        out[:, :, py::2, px::2] = y
    assert (out - ref).abs().max() < 1e-2 * ref.abs().max()  # bf16 rounding of the merged weights
    # the merge itself is exact in fp32
    m = weights.merge_up2x(wt)
    assert torch.allclose(m.sum(dim=(0, 3, 4)) / 4, wt.sum(dim=(2, 3)), atol=1e-4)


def test_fold_layernorm_algebra():
    """LN(x) W^T + b == rstd * (x W'^T - mean * colsum(W')) + (W beta + b) with W' = W diag(gamma) (weights.fold_layernorm), per-row statistics from
    per-32-column {sum, sum of squares} partials as the producer GEMM's epilogue writes them."""
    from ladi_vton_b200 import weights
    g = torch.Generator().manual_seed(3)
    C, N, M = 320, 96, 50
    x = torch.randn(M, C, generator=g) * 2 + 0.5
    W, b = torch.randn(N, C, generator=g) * C ** -0.5, torch.randn(N, generator=g)
    gamma, beta = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g)
    wp, cs, bp = weights.fold_layernorm(W, gamma, beta, b)
    parts = x.view(M, C // 32, 32)
    s, q = parts.sum(-1).sum(-1), (parts * parts).sum(-1).sum(-1)
    mean = s / C
    rstd = torch.rsqrt((q / C - mean * mean).clamp_min(0) + 1e-5)
    got = rstd[:, None] * (x @ wp.float().t() - mean[:, None] * cs[None, :]) + bp
    ref = F.layer_norm(x, (C,), gamma, beta, 1e-5) @ W.t() + b
    assert (got - ref).abs().max() < 2e-2 * ref.abs().max()  # bf16 rounding of W'


def test_pipeline_host_validation_and_signature():
    import inspect
    import ladi_vton_b200 as L
    sig = inspect.signature(L.StableDiffusionTryOnePipeline.__call__)
    want = ["self", "image", "mask_image", "pose_map", "warped_cloth", "prompt", "height", "width", "num_inference_steps", "guidance_scale",
            "negative_prompt", "num_images_per_prompt", "eta", "prompt_embeds", "negative_prompt_embeds", "generator", "latents",
            "output_type", "return_dict", "callback", "callback_steps", "cloth_cond_rate", "no_pose", "cloth_input_type"]
    assert list(sig.parameters)[: len(want)] == want  # tryon_pipe.py:495-520
    d = {k: v.default for k, v in sig.parameters.items()}
    assert (d["num_inference_steps"], d["guidance_scale"], d["eta"], d["output_type"], d["cloth_cond_rate"], d["cloth_input_type"]) == \
        (50, 7.5, 0.0, "pil", 1.0, "warped")
    csig = inspect.signature(L.StableDiffusionTryOnePipeline.__init__)
    assert list(csig.parameters)[1:] == ["vae", "text_encoder", "tokenizer", "unet", "scheduler", "safety_checker", "feature_extractor",
                                         "requires_safety_checker", "emasc", "emasc_int_layers"]  # tryon_pipe.py:56-68
    pipe = L.StableDiffusionTryOnePipeline(vae=L.AutoencoderKL(), text_encoder=None, tokenizer=None, unet=L.UNet2DConditionModel(),
                                           scheduler=L.DDIMScheduler(), emasc=None, emasc_int_layers=None)
    assert pipe.vae_scale_factor == 8
    with pytest.raises(ValueError, match="divisible by 8"):
        pipe.check_inputs(None, 100, 64, 1, None, torch.zeros(1, 77, 8), None)
    with pytest.raises(ValueError, match="Cannot forward both"):
        pipe.check_inputs("a", 64, 64, 1, None, torch.zeros(1, 77, 8), None)
    with pytest.raises(ValueError, match="callback_steps"):
        pipe.check_inputs(None, 64, 64, 0, None, torch.zeros(1, 77, 8), None)
    with pytest.raises(ValueError, match="same shape"):
        pipe.check_inputs(None, 64, 64, 1, None, torch.zeros(1, 77, 8), torch.zeros(2, 77, 8))
    m = torch.tensor([[[[0.2, 0.7], [0.5, 0.49]]]])
    mask, _ = pipe._prepare_mask_and_image(torch.zeros(1, 3, 2, 2), m, None)
    assert m.flatten().tolist() == [0.0, 1.0, 1.0, 0.0] and mask is m  # binarised IN PLACE like the reference
    with pytest.raises(ValueError, match="Image should be"):
        pipe._prepare_mask_and_image(torch.full((1, 3, 2, 2), 2.0), torch.zeros(1, 1, 2, 2), None)
    with pytest.raises(ValueError, match="Mask should be"):
        pipe._prepare_mask_and_image(torch.zeros(1, 3, 2, 2), torch.full((1, 1, 2, 2), 1.5), None)
    # PIL / ndarray branch of prepare_mask_and_masked_image (no EMASC on this pipeline): uint8 RGB -> [-1, 1], L mask -> {0, 1}
    import numpy as np
    from PIL import Image
    im = Image.fromarray(np.full((4, 2, 3), 255, dtype=np.uint8))
    mk = Image.fromarray(np.array([[0, 255], [127, 128], [0, 0], [255, 255]], dtype=np.uint8))
    mask, image = pipe._prepare_mask_and_image(im, mk, None)
    assert image.shape == (1, 3, 4, 2) and float(image.min()) == 1.0 and mask.shape == (1, 1, 4, 2)
    assert mask.flatten().tolist() == [0, 1, 0, 1, 0, 0, 1, 1]
    with pytest.raises(TypeError, match="both"):
        pipe._prepare_mask_and_image(torch.zeros(1, 3, 4, 2), mk, None)
    # generator lists: one (1, ...) draw per sample from its own generator (randn_tensor's list branch)
    from ladi_vton_b200.pipeline import _randn
    gs = [torch.Generator().manual_seed(i) for i in (5, 6)]
    got = _randn((2, 4, 3, 3), gs, torch.device("cpu"))
    want = torch.cat([torch.randn((1, 4, 3, 3), generator=torch.Generator().manual_seed(i)) for i in (5, 6)])
    assert torch.equal(got, want)
    with pytest.raises(ValueError, match="list of generators"):
        _randn((3, 4, 3, 3), [torch.Generator(), torch.Generator()], torch.device("cpu"))
    with pytest.raises(RuntimeError, match="CUDA"):
        pipe.to("cpu")
    with pytest.raises(RuntimeError, match="state_dict mismatch"):
        L.EMASC([64], [64]).load_state_dict({"conv.0.0.weight": torch.zeros(1)})


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    from ladi_vton_b200 import distributed as D
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    total = 5  # ragged on purpose: 3 + 2
    inputs = {"image": torch.arange(total * 6, dtype=torch.float32).reshape(total, 1, 2, 3)}
    mine = D.shard_inputs(inputs, rank, world)
    noise = D.draw_noise(total, 2, 3, torch.Generator().manual_seed(1234))
    mynoise = D.shard_noise(noise, rank, world)
    lo, hi = D.shard_bounds(total, rank, world)
    ok = torch.equal(mynoise[1], noise[1][lo:hi]) and mine["image"].shape[0] == hi - lo
    local = mine["image"].permute(0, 2, 3, 1).repeat(1, 1, 1, 3) + mynoise[0][:, :1].permute(0, 2, 3, 1) * 0  # "images" [b,H,W,3]
    full = D.gather_images(local, world)
    ok = ok and torch.equal(full, inputs["image"].permute(0, 2, 3, 1).repeat(1, 1, 1, 3))
    q.put((rank, bool(ok), (lo, hi)))
    dist.destroy_process_group()


def test_sharding_and_gather_gloo_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
    assert res == [(0, True, (0, 3)), (1, True, (3, 5))]


def test_hub_constructors(tmp_path):
    """hubconf.py:16-66 names and roles; checkpoints come from local files (no network), missing ones fail loudly."""
    import torch
    from ladi_vton_b200 import hub, synthetic as S
    from ladi_vton_b200.vae import EMASC
    with pytest.raises(ValueError):
        hub.extended_unet("viton")
    with pytest.raises(FileNotFoundError, match="unet_vitonhd.pth"):
        hub.extended_unet("vitonhd", checkpoint_dir=str(tmp_path))
    with pytest.raises(FileNotFoundError, match="warping_dresscode.pth"):
        hub.warping_module("dresscode", checkpoint_dir=str(tmp_path))
    ein, eout = [128, 128, 128, 256, 512], [128, 256, 512, 512, 512]
    sd = S.random_state_dict(S.emasc_param_shapes(ein, eout), 3)
    torch.save(sd, tmp_path / "emasc_dresscode.pth")
    m = hub.emasc("dresscode", checkpoint_dir=str(tmp_path))
    assert isinstance(m, EMASC) and sum(v.numel() for v in sd.values()) == 7_965_696
    with pytest.raises(RuntimeError):  # wrong key set -> strict load fails like torch's load_state_dict
        hub.inversion_adapter("vitonhd", state_dict=sd)


def test_coco_body25_mapping_known_answer():
    """src/utils/posemap.py:37-58 (checked equal to the reference dict in the build container): 18 COCO joints, BODY_25 joint 8 skipped."""
    from ladi_vton_b200.data import get_coco_body25_mapping
    m = get_coco_body25_mapping()
    assert len(m) == 18 and [m[i] for i in range(18)] == [0, 1, 2, 3, 4, 5, 6, 7, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18]


def _bench():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_bench_algorithmic_flops_known_answers():
    """bench.py's per-image algorithmic work = SURVEY.md 8(d) / Appendix C (2 flops per MAC of convs, linears, QK^T, PV only):
    15.61 / 33.06 / 62.15 / 120.32 TFLOP at 512x384 for (N, CFG) = (20, off), (50, off), (50, on), (100, on); 79.43 / 173.68 / 330.77 / 644.93
    at 1024x768."""
    bench = _bench()
    want = {(512, 384): (15.61, 33.06, 62.15, 120.32), (1024, 768): (79.43, 173.68, 330.77, 644.93)}
    for (h, w), vals in want.items():
        got = (bench.tflop_per_image(h, w, 20, False), bench.tflop_per_image(h, w, 50, False), bench.tflop_per_image(h, w, 50, True),
               bench.tflop_per_image(h, w, 100, True))
        for g, v in zip(got, vals):
            assert abs(g - v) < 0.02, (h, w, got, vals)  # SURVEY rounds to 2 decimals
    assert bench.tflop_per_image(256, 192, 50, True) < bench.tflop_per_image(512, 384, 50, True)  # other sizes: area-scaled estimate


def test_bench_dump_outputs_whole_or_seeded_sample(tmp_path, monkeypatch):
    """bench.py --dump-outputs: one float32 .npy per output, whole while it fits the size limit; past it, the same seeded sample of its
    elements in every run, and the files stay within the limit."""
    import numpy as np
    bench = _bench()
    x = np.arange(24, dtype=np.float64).reshape(2, 3, 4)
    bench.dump_outputs(str(tmp_path / "a"), {"images": x})
    got = np.load(tmp_path / "a" / "images.npy")
    assert got.dtype == np.float32 and np.array_equal(got, x)
    monkeypatch.setattr(bench, "DUMP_BYTES", 4096 + 400)  # room for 100 float32 values
    big = np.random.default_rng(1).random((50, 60), dtype=np.float32)
    for d in ("b", "c"):
        bench.dump_outputs(str(tmp_path / d), {"images": big})
    b, c = np.load(tmp_path / "b" / "images.npy"), np.load(tmp_path / "c" / "images.npy")
    assert b.shape == (100,) and np.array_equal(b, c) and np.isin(b, big).all()
    assert os.path.getsize(tmp_path / "b" / "images.npy") <= bench.DUMP_BYTES


def test_synthetic_workload_matches_survey_spec():
    """SURVEY.md 8(d): image / cloth ~ U(-1,1), binary centred-rectangle mask over ~35 % of the pixels, 18 Gaussian pose maps (sigma 9,
    exp(-r^2/81)) in [0,1], N(0,1) prompt embeddings [B,77,1024]; seeded (CLI default 1234) and deterministic."""
    from ladi_vton_b200 import synthetic as S
    a, b = S.synthetic_inputs(2, 512, 384), S.synthetic_inputs(2, 512, 384)
    assert all(torch.equal(a[k], b[k]) for k in a)
    assert a["image"].shape == a["warped_cloth"].shape == (2, 3, 512, 384) and float(a["image"].min()) >= -1 and float(a["image"].max()) <= 1
    m = a["mask_image"]
    assert m.shape == (2, 1, 512, 384) and set(m.unique().tolist()) == {0.0, 1.0} and 0.33 < float(m.mean()) < 0.37
    p = a["pose_map"]
    assert p.shape == (2, 18, 512, 384) and float(p.min()) >= 0 and 0.5 < float(p.amax(dim=(2, 3)).min()) <= 1.0
    assert a["prompt_embeds"].shape == a["negative_prompt_embeds"].shape == (2, 77, 1024)
    assert abs(float(a["prompt_embeds"].std()) - 1.0) < 0.02
    assert not torch.equal(S.synthetic_inputs(2, 512, 384, seed=1)["image"], a["image"])


def test_launch_counter_only_counts_real_launches():
    """bench.py's gpu_launches = differences of lib.launches, which lib.call feeds from the library's own counter (ladi_launch_count: incremented
    after every successful cudaLaunchKernelEx).  A call rejected by argument validation launches nothing and must not move either number."""
    from ladi_vton_b200 import lib
    l = lib.load()
    n = l.ladi_launch_count()
    assert n >= 0 and l.ladi_launch_count() == n
    before = lib.launches
    # a count that is not a multiple of 8 is refused before any launch, with or without a device (count 0 is a valid, empty launch)
    with pytest.raises(RuntimeError, match="ladi_add_bf16 failed .*multiple of 8"):
        lib.call("ladi_add_bf16", None, None, None, 7, None)
    assert lib.launches == before and l.ladi_launch_count() == n
