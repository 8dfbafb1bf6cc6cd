#!/usr/bin/env python
"""bench.py -- try-on images/sec of the LaDI-VTON hot path (StableDiffusionTryOnePipeline.__call__) on B200.

One "step" = one pipeline call over one batch of synthetic person/garment/pose/mask tensors with random-init weights
(BASELINE.json configs[1]: VITON-HD shape 512x384, batch 8 per GPU, 50 DDIM steps, bf16, CUDA-graph denoise loop; CLI
default guidance_scale 7.5 => classifier-free guidance on, UNet batch 16 -- SURVEY.md section 8(d)).

  value  : images/sec with the inputs already resident in HBM (device-timed, CUDA events, max over ranks)
  e2e    : images/sec through the public pipeline call with PINNED HOST inputs (H2D) and host numpy outputs (D2H) in the
           timed region
  --impl reference : the reference path's CPU implementation (oracle restatement, fp32, all host threads) on a bounded
           sample of the same workload, extrapolated to images/sec.
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
sys.path.insert(0, ROOT)

# algorithmic 2*MAC counts per image (SURVEY.md Appendix C / BASELINE.md section 3), GFLOP
GF = {(512, 384): dict(unet=581.7, enc=831.1, dec=1879.4, emasc=434.9), (1024, 768): dict(unet=3141.7, enc=3556.1, dec=7749.7, emasc=1739.5)}


def tflop_per_image(H, W, steps, cfg):
    g = GF.get((H, W))
    if g is None:
        s = (H * W) / (512 * 384)
        g = {k: v * s for k, v in GF[(512, 384)].items()}  # attention grows faster; only used for non-baseline sizes
    return (steps * (2 if cfg else 1) * g["unet"] + 2 * g["enc"] + g["dec"] + g["emasc"]) / 1000.0


DUMP_BYTES = 64_000_000  # --dump-outputs writes at most this much, all files together


def dump_outputs(path, arrays):
    """Writes each array as <path>/<name>.npy in float32.  One that would overflow its share of DUMP_BYTES is replaced by a sample of its
    flattened elements at fixed, seeded positions (the same from run to run), so that two builds can be compared file for file."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    share = DUMP_BYTES // len(arrays) - 4096  # room for the .npy header
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float32)
        if a.nbytes > share:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).integers(0, a.size, share // a.itemsize))]
        np.save(os.path.join(path, name + ".npy"), a)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p["bf16_tflops_sustained"], p["bf16_tflops"], p["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 1400.0, 1590.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        self.stop_flag = True
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "power_w_max": max(float(r[2]) for r in self.rows),
                "samples": len(sm), "reasons": reasons}


def cpu_reference_sample(args):
    """The reference's own CPU path (oracle restatement of tryon_pipe.__call__ pieces), fp32, all host threads, on a bounded
    sample: ONE UNet forward of one image's CFG pair (batch 2) + ONE image through VAE encode x2 / EMASC / decode at the
    bench resolution; images/sec = 1 / (ddim_steps * t_unet + t_vae_emasc)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    try:  # keep freed blocks in the heap: without this glibc mmaps/munmaps every large activation and the CPU path spends most
        import ctypes  # of its time in page faults (measured 3x slower)
        libc = ctypes.CDLL("libc.so.6")
        libc.mallopt(-3, 1 << 30)  # M_MMAP_THRESHOLD
        libc.mallopt(-1, 1 << 31)  # M_TRIM_THRESHOLD
    except Exception:
        pass
    import torch
    import torch.nn.functional as F  # noqa: F401
    from ladi_oracle.parts import EMASC, mask_features
    from ladi_oracle.unet import UNet2DConditionModel as OU
    from ladi_oracle.vae import AutoencoderKL as OV
    from ladi_vton_b200 import synthetic as S
    from ladi_vton_b200.unet import unet_param_shapes
    from ladi_vton_b200.vae import vae_param_shapes
    # thread count: PINNED to min(64, host threads).  On these layer sizes PyTorch's CPU kernels get slower past ~64 threads (sync
    # overhead; measured in round 1 on the 128-thread GPU-box hosts), and a per-run calibration made the arm swing 6x between runs.
    best = max(1, min(64, os.cpu_count() or 1))
    torch.set_num_threads(best)
    args.cpu_threads = best
    cfg = args.guidance > 1.0
    H, W = args.height, args.width
    with torch.no_grad():
        with torch.device("meta"):  # skip nn.Module default init of 950 M parameters; weights are assigned below
            ou, ov, oe = OU().eval(), OV().eval(), EMASC(S.EMASC_IN, S.EMASC_OUT).eval()
        ou.load_state_dict(S.random_state_dict(unet_param_shapes({}), 1234, fast=True), assign=True)
        ov.load_state_dict(S.random_state_dict(vae_param_shapes({}), 1235, fast=True), assign=True)
        oe.load_state_dict(S.random_state_dict(S.emasc_param_shapes(S.EMASC_IN, S.EMASC_OUT), 1236), assign=True)
        inp = S.synthetic_inputs(1, H, W)
        bp = 2 if cfg else 1
        x = torch.randn(bp, 31, H // 8, W // 8)
        ctx = torch.cat([inp["negative_prompt_embeds"], inp["prompt_embeds"]]) if cfg else inp["prompt_embeds"]

        def sample():
            t0 = time.perf_counter()
            ou(x, torch.tensor(501), ctx)
            t1 = time.perf_counter()
            ov.encode(inp["warped_cloth"])
            enc, feats = ov.encode(inp["image"] * (inp["mask_image"] < 0.5))
            inter = mask_features(oe([feats[i] for i in range(1, 6)]), inp["mask_image"])
            ov.decode(enc.latent_dist.mode(), list(inter), [1, 2, 3, 4, 5])
            t2 = time.perf_counter()
            return t1 - t0, t2 - t1
        return sample


def run_reference(args, rank):
    if rank != 0:
        return
    import torch
    t_start = time.perf_counter()
    sample = cpu_reference_sample(args)
    budget = 270.0  # seconds for warm-up + timed samples: the whole arm must end within a few minutes whatever K / W are
    done_w = 0
    for _ in range(args.warmup):
        if done_w >= 1 and (time.perf_counter() - t_start) > budget * 0.4:
            break
        sample()
        done_w += 1
    tu, tv, done = 0.0, 0.0, 0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        a, b = sample()
        tu, tv, done = tu + a, tv + b, done + 1
        if (time.perf_counter() - t_start) > budget:
            break
    wall = time.perf_counter() - t0
    tu, tv = tu / done, tv / done
    args.steps_done, args.warmup_done = done, done_w
    per_image = args.ddim_steps * tu + tv
    v = 1.0 / per_image
    cores = getattr(args, "cpu_threads", os.cpu_count())
    line = {"metric": "try-on images/sec", "value": v, "unit": "images/s", "impl": "reference", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": wall / args.steps_done * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "steps_completed": args.steps_done, "warmup_completed": args.warmup_done, "dtype": "fp32", "data": "synthetic",
            "config": dict(workload_config(args), reference_sample=f"what this arm actually executes: batch 1 (UNet batch {2 if args.guidance > 1 else 1}), fp32, "
                           f"ONE UNet forward + one image through VAE enc x2 / EMASC / dec per step, images/s extrapolated to {args.ddim_steps} DDIM steps; "
                           f"{cores} host threads (pinned)"),
            "cpu_baseline": {"value": v, "unit": "images/s", "cores": cores, "kind": "port",
                             "sample": f"1 UNet fwd (batch {2 if args.guidance > 1 else 1}) {tu:.2f}s + 1 image VAE enc x2/EMASC/dec {tv:.2f}s per step; "
                                       f"extrapolated to {args.ddim_steps} DDIM steps; torch {torch.__version__} fp32, {cores} of {os.cpu_count()} host threads (pinned: min(64, host threads))"},
            "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def workload_config(args):
    cfg = args.guidance > 1.0
    return {"workload": f"VITON-HD shape {args.height}x{args.width}, batch {args.batch}/GPU, {args.ddim_steps} DDIM steps, "
                        f"guidance_scale {args.guidance} ({'CFG on: UNet batch ' + str(2 * args.batch) if cfg else 'no CFG'}), bf16, CUDA-graph denoise loop",
            "global_batch": args.batch * args.gpus, "height": args.height, "width": args.width, "ddim_steps": args.ddim_steps,
            "guidance_scale": args.guidance, "parallelism": f"dp{args.gpus} (batch-sharded replicas, NCCL all_gather of the uint8 images)",
            "l2": "working set (1.9 GB bf16 weights per UNet forward) >> 126 MB L2; no flush needed"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--batch", type=int, default=8, help="images per GPU")
    ap.add_argument("--height", type=int, default=512)
    ap.add_argument("--width", type=int, default=384)
    ap.add_argument("--ddim-steps", type=int, default=50)
    ap.add_argument("--guidance", type=float, default=7.5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the images the last timed step returned as DIR/images.npy "
                    "(float32; with --gpus > 1 the gathered uint8 batch as 0..255)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "engine":
        ap.error("--dump-outputs needs --impl engine: the reference arm times a sample of the work and returns no images")
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        return run_reference(args, rank)

    import torch
    import torch.distributed as dist
    from ladi_vton_b200 import lib, ops, synthetic as S
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    cfg = args.guidance > 1.0
    B, H, W = args.batch, args.height, args.width
    pipe, _ = S.build_pipeline(dev, weights_on_device=True)  # full-size random-init UNet (865,988,484 params) / VAE / EMASC
    host = S.synthetic_inputs(B, H, W, seed=1234 + rank)
    pinned = {k: v.pin_memory() for k, v in host.items()}
    resident = {k: v.to(dev) for k, v in host.items()}
    gen = torch.Generator(device=dev).manual_seed(1234)
    gather = torch.empty((world * B, H, W, 3), dtype=torch.uint8, device=dev) if world > 1 else None  # numpy_to_pil's uint8, 0.59 MB / image
    host_all = torch.empty((world * B, H, W, 3), dtype=torch.uint8, pin_memory=True) if (world > 1 and rank == 0) else None

    def call(inputs, output_type):
        out = pipe(image=inputs["image"], mask_image=inputs["mask_image"], pose_map=inputs["pose_map"], warped_cloth=inputs["warped_cloth"],
                   prompt_embeds=inputs["prompt_embeds"], negative_prompt_embeds=inputs["negative_prompt_embeds"], height=H, width=W,
                   num_inference_steps=args.ddim_steps, guidance_scale=args.guidance, generator=gen, output_type=output_type).images
        return out

    last = {}

    def step_resident():
        img = call(resident, "pt_u8" if world > 1 else "pt")
        if world > 1:
            dist.all_gather_into_tensor(gather, img)  # the path's only collective: final image gather over NVLink
        last["images"] = gather if world > 1 else img

    def step_e2e():
        dev_in = {k: v.to(dev, non_blocking=True) for k, v in pinned.items()}  # H2D from pinned host memory
        if world > 1:  # every rank: H2D of its shard -> pipeline -> uint8 gather; rank 0: D2H of the whole batch into pinned memory
            img = call(dev_in, "pt_u8")
            dist.all_gather_into_tensor(gather, img)
            if rank == 0:
                host_all.copy_(gather, non_blocking=True)
                torch.cuda.current_stream().synchronize()
                return host_all.numpy()
            return None
        return call(dev_in, "np")  # D2H (pinned staging) inside

    def timed(fn, warmup, steps):
        for _ in range(warmup):
            fn()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = lib.launches
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item() / steps, (lib.launches - n0)

    sampler = ClockSampler(local)
    sampler.start()
    ms_step, launches = timed(step_resident, args.warmup, args.steps)
    clocks = sampler.summary()
    if args.dump_outputs and rank == 0:  # before the e2e pass: it writes into the same gather buffer
        dump_outputs(args.dump_outputs, {k: v.float().cpu().numpy() for k, v in last.items()})
    ms_e2e, _ = timed(step_e2e, 1, args.steps)

    # ---- roofline of the dominant kernel: one instrumented eager UNet forward, every conv/GEMM launch bracketed by CUDA events
    sustained, burst, hbm, src = peaks()
    ops.PROFILE = []
    s = next(iter(pipe._sessions.values()))
    pipe.unet._ctx = s.ctx_kv
    pipe.unet.forward_nhwc(s.unet_in, s.step)
    torch.cuda.synchronize()
    conv = [(e0.elapsed_time(e1), fl) for (name, e0, e1, fl, _) in ops.PROFILE if name == "ladi_conv2d_bf16"]
    attn = [(e0.elapsed_time(e1), fl) for (name, e0, e1, fl, _) in ops.PROFILE if name == "ladi_attention_bf16"]
    allk = sum(e0.elapsed_time(e1) for (_, e0, e1, _, _) in ops.PROFILE)
    ops.PROFILE = None
    t_conv, f_conv = sum(t for t, _ in conv), sum(f for _, f in conv)
    t_attn, f_attn = sum(t for t, _ in attn), sum(f for _, f in attn)
    ach = f_conv / (t_conv * 1e-3) / 1e12
    # the same launches INSIDE the replayed step graph (what the timed region runs): kernel durations from one CUPTI-traced replay
    # (torch.profiler), outside the timed region.  Reported beside the event-bracketed eager figure, never instead of it.
    in_graph = None
    try:
        from torch.profiler import ProfilerActivity, profile
        s.step.zero_()
        s.g_step.replay(); torch.cuda.synchronize()
        s.step.zero_()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            s.g_step.replay()
            torch.cuda.synchronize()
        ev = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "Memcpy" not in e.name and "Memset" not in e.name),
                    key=lambda e: e.time_range.start)
        # exclusive time per kernel: with programmatic dependent launch a kernel's CTAs start (and wait) while its predecessor drains;
        # only the part after the predecessor's end is attributed to it, so the family sums add up to the step's wall time
        fam = {"conv": 0.0, "attention": 0.0, "norm": 0.0, "other": 0.0}
        prev_end = None
        for e in ev:
            st = e.time_range.start if prev_end is None else max(e.time_range.start, prev_end)
            d = max(0.0, e.time_range.end - st) * 1e-3  # ms
            k = ("conv" if ("convgemm_kernel" in e.name or "splitk_reduce" in e.name) else "attention" if "attention_" in e.name
                 else "norm" if ("gn_" in e.name or "layernorm" in e.name) else "other")
            fam[k] += d
            prev_end = e.time_range.end if prev_end is None else max(prev_end, e.time_range.end)
        wall = (prev_end - ev[0].time_range.start) * 1e-3
        in_graph = {"conv_ms": fam["conv"], "attention_ms": fam["attention"], "norm_ms": fam["norm"], "other_ms": fam["other"], "kernels": len(ev),
                    "step_wall_ms": wall, "conv_tflops": f_conv / (fam["conv"] * 1e-3) / 1e12 if fam["conv"] else None,
                    "attention_tflops": f_attn / (fam["attention"] * 1e-3) / 1e12 if fam["attention"] else None,
                    "unet_forward_tflops": (f_conv + f_attn) / (wall * 1e-3) / 1e12}
    except Exception as e:  # the profiler is evidence, not the product: never fail the bench on it
        in_graph = {"error": repr(e)[:200]}
    roofline = {"bound": "tensor", "kernel": "convgemm_kernel (implicit-GEMM conv + linear, tcgen05 cta_group::2 CTA pairs)", "achieved": ach, "peak": sustained,
                "unit": "TFLOP/s", "frac": ach / sustained, "peak_source": src + ", sustained bf16",
                "how": "achieved = sum of algorithmic 2*M*N*K over the conv/GEMM launches of ONE UNet forward / sum of their CUDA-event durations, "
                       "each launch bracketed on torch's current stream in an eager (un-graphed) forward after the timed region; "
                       "in_graph = the same launches inside the replayed step graph, durations from a CUPTI trace of one replay",
                "in_graph": in_graph, "frac_in_graph": (in_graph["conv_tflops"] / sustained) if in_graph and in_graph.get("conv_tflops") else None,
                "traffic": None, "traffic_note": None,
                "launches_per_unet_forward": len(conv), "avg_launch_ms": t_conv / max(1, len(conv)),
                "algorithmic_gflop_per_launch": f_conv / max(1, len(conv)) / 1e9, "share_of_unet_forward": t_conv / allk}
    # per-launch DRAM traffic of the dominant kernel: only from a COMMITTED ncu capture of this very workload (profiles/r02_ncu_traffic.json,
    # written by tools/ncu_traffic.py from `ncu --set full`), matched on the workload key; otherwise null -- never a constant from another run
    try:
        with open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")) as f:
            tj = json.load(f)
        if tj.get("workload_key") == [B, H, W, bool(cfg)]:
            roofline["traffic"] = tj["avg_dram_bytes_per_launch"]
            roofline["traffic_note"] = tj["note"]
    except Exception:
        pass
    attention_roofline = {"bound": "tensor (MUFU-limited softmax at head_dim 64)", "kernel": "attention_pair_kernel / attention_single_kernel (flash, tcgen05 + TMEM)",
                          "achieved": f_attn / (t_attn * 1e-3) / 1e12 if t_attn else None, "peak": sustained, "unit": "TFLOP/s",
                          "frac": (f_attn / (t_attn * 1e-3) / 1e12 / sustained) if t_attn else None,
                          "achieved_in_graph": in_graph.get("attention_tflops") if in_graph else None,
                          "share_of_unet_forward": t_attn / allk, "launches": len(attn),
                          "algorithmic_gflop_per_forward": f_attn / 1e9}

    if rank == 0:
        imgs = B * world
        value = imgs / (ms_step * 1e-3)
        e2e = imgs / (ms_e2e * 1e-3)
        tf_img = tflop_per_image(H, W, args.ddim_steps, cfg)
        h2d = sum(v.numel() * v.element_size() for v in pinned.values())
        line = {"metric": "try-on images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": workload_config(args), "clocks": clocks, "gpu_launches": launches,
                "e2e": {"value": e2e, "unit": "images/s", "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": (B * world * H * W * 3) if world > 1 else (B * H * W * 3 * 4),  # N>1: rank 0 reads the gathered uint8 batch; N=1: fp32 numpy
                        "ms_per_step": ms_e2e},
                "roofline": roofline, "roofline_attention": attention_roofline,
                "pipeline_tensor_frac": value * tf_img / (sustained * world), "tflop_per_image": tf_img}
        if world == 1 and not args.no_cpu_baseline:
            sample = cpu_reference_sample(args)
            tu, tv = sample()
            if tu + tv < 30.0:  # first sample doubles as warm-up when a second one is affordable
                tu, tv = sample()
            v = 1.0 / (args.ddim_steps * tu + tv)
            line["cpu_baseline"] = {"value": v, "unit": "images/s", "cores": getattr(args, "cpu_threads", os.cpu_count()), "kind": "port",
                                    "sample": f"1 UNet fwd (batch {2 if cfg else 1}) {tu:.2f}s + 1 image VAE enc x2/EMASC/dec {tv:.2f}s on the host CPU, "
                                              f"extrapolated to {args.ddim_steps} DDIM steps (oracle restatement, fp32, {getattr(args, 'cpu_threads', 0)} of {os.cpu_count()} host threads)"}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
