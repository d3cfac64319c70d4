#!/usr/bin/env python
"""bench.py — SeedVR2-3B upscaled frames/s on B200 (BASELINE.json metric).

    python bench.py [--gpus N --steps K --warmup W] [--workload 4k_shard|1080p|...] [--impl reference]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path (VAE encode -> DiT one-step -> VAE decode)
over one clip of synthetic video per GPU.  Default workload = the per-GPU shard
of BASELINE config 3 (8 frames, padded to 9, 720p->4K at 2160x3840): at N GPUs
every rank processes its own clip (weak scaling, the reference's data-parallel
partition by clip, inference_cli.py:1161-1193) and one NCCL all-gather returns
the decoded frames.  Output: ONE JSON line on rank 0 (see the task contract).

  value : frames/s, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e   : same through SeedVR2Engine.upscale_clip with pinned HOST input frames
          (H2D inside the timed region) and the result read back to host (D2H)
  roofline : the tcgen05 GEMM/implicit-conv kernel (dominant): algorithmic FLOPs of
          all its launches / their CUDA-event time, vs the measured bf16 peak
  cpu_baseline : the oracle port (torch fp32, all host threads) on a bounded sample

--dump-outputs DIR writes what the last timed step of `value` returned (rank 0) as DIR/<name>.npy in float32, so that
two builds can be compared output for output on identical seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

# the tree the benchmark runs from may be read-only: no bytecode caches written next to the sources
sys.dont_write_bytecode = True

# Clips that fill the HBM (temporally sliced VAE passes sized from the free memory) need an allocator that does not
# fragment: expandable segments, chosen before torch initialises CUDA.  The default workloads keep torch's default.
if any(("4k_clip64" in a or "vae_decode" in a) for a in sys.argv):
    os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")

import torch  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (real frames, H, W, description)
    "4k_shard": (8, 2160, 3840, "SeedVR2-3B bf16, 8-frame (->9) 720p->4K clip per GPU = BASELINE config 3 shard"),
    "1080p": (16, 1080, 1920, "SeedVR2-3B bf16, 16-frame (->17) 540p->1080p clip = BASELINE config 2"),
    "4k_clip64": (64, 2160, 3840, "SeedVR2-3B bf16, 64-frame (->65) 720p->4K as ONE clip on one GPU = BASELINE config 3' "
                                  "(17 latent frames, 2083-token windows, temporally sliced VAE)"),
    "4k_shard_7b": (4, 2160, 3840, "SeedVR2-7B bf16, 4-frame (->5) 720p->4K clip per GPU = BASELINE config 4 shard"),
    "image_512": (1, 512, 512, "SeedVR2-3B bf16, one 256x256 -> 512x512 image = BASELINE config 1"),
    "720p": (8, 720, 1280, "SeedVR2-3B bf16, 8-frame (->9) 360p->720p clip (smoke)"),
    "tiny": (4, 128, 192, "tiny clip (smoke)"),
}
# BASELINE config 5: VAE-only decode of a latent (T, 90, 160) -> (4T-3) frames of 720 x 1280, `--workload vae_decode_T<T>`
for _t in (16, 32, 64, 128):
    WORKLOADS[f"vae_decode_T{_t}"] = (4 * _t - 3, 720, 1280, f"VAE-only 3D-conv decode, latent T={_t} x 90 x 160 -> "
                                                               f"{4 * _t - 3} frames 720x1280 = BASELINE config 5")
DEFAULT_WORKLOAD = "4k_shard"


def flop_model(frames_pad: int, H: int, W: int, variant="3b"):
    """BASELINE.md §2 work model (FLOP = 2 MAC)."""
    Hp, Wp = (H + 15) // 16 * 16, (W + 15) // 16 * 16
    T_lat, h, w = (frames_pad - 1) // 4 + 1, Hp // 8, Wp // 8
    L = T_lat * (h // 2) * (w // 2)
    n = h * w
    per_tok = 5.075e9 if variant == "3b" else 8.15e9
    attn_vae = T_lat * (4.0 * n * n * 512 + 8.0 * n * 512 * 512)
    return dict(dit=per_tok * L, enc=9.0e6 * frames_pad * Hp * Wp + attn_vae,
                dec=24.2e6 * frames_pad * Hp * Wp + attn_vae, tokens=L)


DUMP_SAMPLE = 8 * 2**20         # elements kept of an output larger than that: 32 MiB of float32 per array


def dump_outputs(path, arrays):
    """Each tensor as path/<name>.npy in float32: whole when it has at most DUMP_SAMPLE elements, else the elements at
    DUMP_SAMPLE sorted flat indices drawn from a fixed seed (the same positions for every build of one workload)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_SAMPLE:
            idx = torch.randint(t.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(path, f"{name}.npy"), t.float().cpu().numpy())


def synth_frames(T, H, W, seed=42, device="cpu"):
    """Low-res noise field bicubic-upsampled + 2 % white noise (SURVEY.md §8(d))."""
    g = torch.Generator().manual_seed(seed)
    lo = torch.rand(T, 3, max(H // 8, 2), max(W // 8, 2), generator=g)
    x = torch.nn.functional.interpolate(lo, size=(H, W), mode="bicubic", align_corners=False)
    x = (x + 0.02 * torch.randn(x.shape, generator=g)).clamp(0, 1)
    return x.permute(0, 2, 3, 1).contiguous().to(device)       # T,H,W,3


class ClockSampler(threading.Thread):
    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag = index, [], set(), False
        self.max_mhz = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                f = [s.strip() for s in out.split(",")]
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for nme, v in zip(names, f[2:]):
                    if v.lower().startswith("active"):
                        self.reasons.add(nme)
            except Exception:
                pass
            time.sleep(0.2)

    def result(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ----------------------------------------------------------------------------
# CPU baseline: the oracle port on host cores, bounded sample, extrapolated by the FLOP model
# ----------------------------------------------------------------------------
def cpu_oracle_sample(frames_pad, H, W, seconds_budget=25.0):
    from oracle import dit_oracle, vae_oracle
    from svr2_import import load_package
    pkg = load_package()
    # torch's CPU conv/GEMM scale poorly past a few dozen threads on samples this small
    torch.set_num_threads(min(os.cpu_count() or 1, 32))
    cores = torch.get_num_threads()
    t_all = time.time()
    # VAE sample: full-width VAE, 5 frames of 96x128 (one untimed warm-up on a tiny clip first)
    sdv = {k: v.float() for k, v in pkg.weights.synth_vae_state_dict(seed=4321).items()}
    g = torch.Generator().manual_seed(0)
    vae_oracle.vae_decode(sdv, vae_oracle.vae_encode(sdv, torch.rand(1, 3, 1, 32, 32, generator=g)))
    x = torch.rand(1, 3, 5, 96, 128, generator=g) * 2 - 1
    t0 = time.time(); z = vae_oracle.vae_encode(sdv, x); t_enc = time.time() - t0
    t0 = time.time(); vae_oracle.vae_decode(sdv, z); t_dec = time.time() - t0
    fm_s = flop_model(5, 96, 128)
    enc_rate, dec_rate = fm_s["enc"] / t_enc, fm_s["dec"] / t_dec
    del sdv
    # DiT sample: 3B width, 2 layers (1 specific + 1 shared/last), 3x20x36 tokens
    cfg = dit_oracle.dit_config("3b", layers=2, mm_layers=1)
    sdd = {k: v.float() for k, v in pkg.weights.synth_dit_state_dict(cfg, seed=1).items()}
    T, Hl, Wl = 3, 48, 80
    vid = torch.randn(T * Hl * Wl, 33, generator=g)
    txt = torch.randn(58, 5120, generator=g)
    dit_oracle.dit_forward(sdd, cfg, vid[: 1 * 8 * 8], txt, 1, 8, 8)          # untimed warm-up
    t0 = time.time(); dit_oracle.dit_forward(sdd, cfg, vid, txt, T, Hl, Wl); t_dit = time.time() - t0
    dit_rate = (158.6e6 * 2 * T * (Hl // 2) * (Wl // 2)) / t_dit
    fm = flop_model(frames_pad, H, W)
    est_s = fm["enc"] / enc_rate + fm["dec"] / dec_rate + fm["dit"] / dit_rate
    return dict(cores=cores, est_clip_seconds=est_s, rates_gflops=dict(enc=enc_rate / 1e9, dec=dec_rate / 1e9,
                dit=dit_rate / 1e9), sample_seconds=time.time() - t_all,
                sample="oracle (torch fp32) on host: full-width VAE encode+decode of 5x96x128 px, 3B-width DiT "
                       "2 layers on 2880 tokens; clip time extrapolated with the BASELINE.md FLOP model")


def run_reference_arm(args, frames_real, frames_pad, H, W, workload_desc):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals = []
    info = None
    for i in range(args.warmup + args.steps):
        info = cpu_oracle_sample(frames_pad, H, W)
        if i >= args.warmup:
            vals.append(frames_real / info["est_clip_seconds"])
    v = sum(vals) / len(vals)
    metric = "upscaled frames/sec SeedVR2-3B 720p->4K" if args.workload == "4k_shard" else "upscaled frames/sec SeedVR2-3B"
    line = {"metric": metric, "value": v, "unit": "frames/s", "impl": "reference",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * frames_real / v, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_desc, "note": "reference PyTorch path restated by oracle/ (the reference "
                       "itself cannot be installed: diffusers/omegaconf/rotary_embedding_torch absent); CPU fp32"},
            "extrapolated": True,
            "cpu_baseline": {"value": float(f"{v:.2g}"), "unit": "frames/s", "cores": info["cores"], "kind": "port",
                             "extrapolated": True, "sample": info["sample"]},
            "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------
# per-kernel table: C-ABI entry point -> (bound, what the profiler's flops / bytes annotation means)
HBM_KERNELS = {"svr2_groupnorm_from_stats_bf16", "svr2_groupnorm_bf16", "svr2_rmsnorm_ada_bf16", "svr2_conv_tap_gather",
               "svr2_qk_norm_rope_window_bf16", "svr2_resize_bicubic_aa_bf16", "svr2_sample_to_image_bf16",
               "svr2_txt_window_mean_bf16", "svr2_im2col3_bf16", "svr2_ncdhw_to_ndhwc_bf16", "svr2_transpose_bf16"}


def kernel_table(prof, steps, peak_tf, peak_gbs, step_ms):
    """[{name, ms, share, bound, achieved, unit, frac}] per C-ABI entry point, largest first (algorithmic FLOPs or bytes
    of all its launches / their CUDA-event time, against the measured tensor / HBM peak)."""
    agg = {}
    for n, d in prof.items():
        a = agg.setdefault(n.split("|")[0], dict(ms=0.0, flops=0.0, bytes=0.0, calls=0))
        for k in ("ms", "flops", "bytes", "calls"):
            a[k] += d[k]
    rows = []
    for n, a in sorted(agg.items(), key=lambda kv: -kv[1]["ms"]):
        row = {"name": n, "calls_per_step": a["calls"] // steps, "ms": round(a["ms"] / steps, 3),
               "share": round(a["ms"] / steps / step_ms, 4)}
        if a["flops"] > 0:
            ach = a["flops"] / a["ms"] / 1e9
            row.update(bound="tensor", achieved=round(ach, 1), unit="TFLOP/s", frac=round(ach / peak_tf, 3))
        elif a["bytes"] > 0:
            ach = a["bytes"] / a["ms"] / 1e6
            row.update(bound="hbm", achieved=round(ach, 1), unit="GB/s", frac=round(ach / peak_gbs, 3))
        else:
            row.update(bound="hbm" if n in HBM_KERNELS else "latency", achieved=None, unit=None, frac=None)
        rows.append(row)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--lib-baseline", default="default", choices=["none", "ops", "default", "full"],
                    help="time the reference's GPU libraries beside the engine (tools/gpu_library_baseline.py): ops = "
                         "flash-attn-2 / SDPA, cuBLAS, cuDNN on the 4K-shard shapes; default = ops + the reference's bf16 "
                         "library flow per phase at BASELINE config 2; full = + the 4K shard (N = 1, rank 0 only)")
    ap.add_argument("--source", default="lowres", choices=["lowres", "target"],
                    help="lowres: the clip enters at its source resolution (H/3 x W/3 for 720p->4K, H/2 x W/2 for "
                         "540p->1080p) and is resized on the device by the pre-processing kernel, as in the "
                         "reference pipeline; target: frames already at the target resolution")
    ap.add_argument("--no_graph", action="store_true",
                    help="time the end-to-end region with eager launches instead of one CUDA-graph replay per clip")
    ap.add_argument("--color_correction", default="none", choices=["none", "lab", "wavelet", "adain"],
                    help="post-decode colour correction inside the step (reference CLI default: lab); the headline "
                         "metric is quoted with 'none' = the north_star path (encode + DiT + decode)")
    ap.add_argument("--phases", action="store_true", help="print a per-kernel breakdown to stderr")
    ap.add_argument("--detail", action="store_true", help="with --phases: break GEMM/conv launches down by shape")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned to DIR/<name>.npy (float32; a fixed, seeded sample "
                         f"of {DUMP_SAMPLE} elements of a larger output)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    frames_real, H, W, desc = WORKLOADS[args.workload]
    vae_only = args.workload.startswith("vae_decode")
    from svr2_import import load_package
    pkg = load_package()
    import importlib
    pipeline = importlib.import_module("comfyui_seedvr2_videoupscaler_b200.pipeline")
    frames_pad = pipeline.pad_4n1(frames_real)

    if args.impl == "reference":
        return run_reference_arm(args, frames_real, frames_pad, H, W, desc)

    lib = importlib.import_module("comfyui_seedvr2_videoupscaler_b200.lib")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    variant = "7b" if args.workload.endswith("_7b") else "3b"
    eng = pipeline.build_synthetic_engine(variant, device=dev)
    # source clip: 720p for the 4K shard (x3), 540p for 1080p (x2), half size otherwise
    div = 1 if (args.source == "target" or vae_only) else (3 if H == 2160 else 2)
    if vae_only:        # config 5: the step is one decode of a synthetic latent (T, 90, 160, 16), scaled like the runner's
        T_lat = (frames_real + 3) // 4
        g = torch.Generator().manual_seed(42 + rank)
        frames_host = (torch.randn(T_lat, H // 8, W // 8, 16, generator=g) * 0.9152).to(torch.bfloat16).pin_memory()
        out_host = torch.empty(3, frames_real, H, W, dtype=torch.bfloat16).pin_memory()
    else:
        frames_host = synth_frames(frames_real, H // div, W // div, seed=42 + rank).to(torch.bfloat16).pin_memory()
        out_host = torch.empty(frames_real, H, W, 3, dtype=torch.bfloat16).pin_memory()
    frames_dev = frames_host.to(dev)
    gather_buf = torch.empty((world,) + tuple(out_host.shape), device=dev, dtype=torch.bfloat16) if world > 1 else None
    # a buffer larger than L2 (126 MB) written between steps is unnecessary: every step streams > 10 GB of activations
    noise = None

    def step(src):
        if vae_only:
            y = eng.vae_decode(src)
        else:
            y = eng.upscale_clip(src, noise=noise, seed=42, color_correction=args.color_correction, resolution=H)
        if world > 1:
            dist.all_gather_into_tensor(gather_buf.view(-1), y.reshape(-1).contiguous())
        return y

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step(frames_dev)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # ---- timed region A: inputs resident in HBM, the product path (encode / DiT / decode sequenced by the native C++
    # runtime in ONE planned workspace per clip), eager launches
    torch.cuda.reset_peak_memory_stats()
    lib.LAUNCHES = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        y = step(frames_dev)
        if i + 1 < args.steps:          # only the last step's result stays alive
            del y
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = lib.LAUNCHES
    peak_mem_native = torch.cuda.max_memory_allocated()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"sample" if vae_only else "frames": y})
    del y
    # ---- region P: the same steps with per-kernel CUDA events on the launching stream (per-call events need the Python
    # sequencing of the same kernels): the roofline and the per-kernel table come from here, not the headline value
    prof_steps = 1 if ms / args.steps > 5000 else min(args.steps, 3)      # long clips: one profiled pass is enough
    lib.release_workspace(dev)      # the call-by-call sequencing allocates per activation: it needs the resident block's bytes
    lib.PROFILER = lib.Profiler()   # (set BEFORE the warm pass: with no profiler the step would run natively and re-create the block)
    lib.PROFILER.detail = args.detail
    step(frames_dev)            # the Python sequencing allocates per activation: first pass fills the allocator's cache
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    lib.PROFILER.reset()
    p0.record()
    for _ in range(prof_steps):
        step(frames_dev)
    p1.record()
    barrier()
    ms_prof = p0.elapsed_time(p1)
    prof = lib.PROFILER.summary()
    lib.PROFILER = None
    # ---- "DiT step ms" (BASELINE.json metric, second half): one NaDiT forward (+ the x0 = noise - v endpoint) at this
    # workload's latent geometry, CUDA events, inputs resident
    dit_step_ms = None
    if not vae_only:
        lshape = eng.latent_shape(frames_dev, H)
        lat = torch.randn(lshape, device=dev, dtype=torch.bfloat16)
        nz = torch.randn(lshape, device=dev, dtype=torch.bfloat16)
        eng.inference(nz, lat)
        torch.cuda.synchronize()
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        d0.record()
        for _ in range(3):
            eng.inference(nz, lat)
        d1.record()
        torch.cuda.synchronize()
        dit_step_ms = d0.elapsed_time(d1) / 3
        del lat, nz
    # ---- timed region B: end to end with host buffers.  On one GPU the clip is replayed as ONE CUDA graph
    # (SeedVR2Engine.graphed: same kernels, same results, no per-launch host work, so a busy host cannot stall the
    # GPU); any capture problem falls back to eager launches and is reported in the JSON line.
    graphed, graph_note = None, "eager launches"
    if world == 1 and not args.no_graph and not vae_only:
        try:
            graphed = eng.graphed(frames_dev, seed=42, warmup=0, color_correction=args.color_correction, resolution=H)
            graph_note = "CUDA-graph replay of the clip"
        except Exception as ex:   # noqa: BLE001 - the harness must still produce its line
            graphed, graph_note = None, f"eager launches (graph capture failed: {type(ex).__name__})"
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if graphed is not None:                   # one untimed replay: first-replay graph upload is not steady state
        graphed(frames_host.to(dev, non_blocking=True))
        torch.cuda.synchronize()
    else:                                     # eager: one untimed step re-creates the engine's resident workspace (released for
        step(frames_host.to(dev, non_blocking=True))      # the profiled region) outside the timed region
        torch.cuda.synchronize()
    e2.record()
    for _ in range(args.steps):
        src = frames_host.to(dev, non_blocking=True)
        y = graphed(src) if graphed is not None else step(src)
        out_host.copy_(y, non_blocking=True)
    e3.record()
    barrier()
    ms_e2e = e2.elapsed_time(e3)
    sampler.stop_flag = True
    peak_mem = torch.cuda.max_memory_allocated()
    del graphed
    torch.cuda.empty_cache()

    t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = t.tolist()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    total_frames = frames_real * world * args.steps
    value = total_frames / (ms / 1e3)
    e2e = total_frames / (ms_e2e / 1e3)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_gbs = peaks.get("hbm_gbs", 6500.0)
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks else "fallback 1.4 PFLOP/s sustained (of fallback)"
    gemm_names = ("svr2_linear_bf16", "svr2_linear_ex_bf16", "svr2_linear_qkv_rope_bf16", "svr2_conv3d_bf16",
                  "svr2_conv3d_stats_bf16", "svr2_conv3d_shortcut_stats_bf16", "svr2_upsample_shuffle_bf16")
    is_gemm = lambda n: n.split("|")[0] in gemm_names
    g_flops = sum(d["flops"] for n, d in prof.items() if is_gemm(n))
    g_ms = sum(d["ms"] for n, d in prof.items() if is_gemm(n))
    g_calls = sum(d["calls"] for n, d in prof.items() if is_gemm(n))
    achieved = g_flops / (g_ms / 1e3) / 1e12 if g_ms > 0 else 0.0
    fm = flop_model(frames_pad, H, W, variant)
    # DRAM traffic of the dominant kernel: NOT measured in this run (that needs ncu) — taken from the committed
    # `ncu --set full` capture of one representative launch and labelled as such; null when the workload does not run it
    traffic, traffic_detail = None, None
    try:
        cap_file = next(f for f in ("ncu_full_r2.json", "ncu_full_r1.json") if os.path.exists(os.path.join(ROOT, "profiles", f)))
        cap = json.load(open(os.path.join(ROOT, "profiles", cap_file)))["conv256_pair"]
        if H >= 1080 and not args.workload.startswith("image"):
            traffic = (float(cap["dram__bytes_read.sum"]) + float(cap["dram__bytes_write.sum"])) * 1e9   # bytes per launch
            traffic_detail = {"source": f"static: profiles/{cap_file} (ncu --set full of one launch, not this run)",
                              "algorithmic_bytes_per_launch": (4 + 2) * 1080 * 1920 * 256 * 2.0,
                              "launch": "conv3d 256->256 3x3x3, 2 frames 1080x1920 (+2 halo frames)",
                              "tensor_pipe_active_pct": float(cap["sm__mem_tensor_cycles_active.avg.pct_of_peak_sustained_elapsed"])}
    except Exception:
        pass
    if args.phases:
        tot = sum(d["ms"] for d in prof.values())
        for n, d in sorted(prof.items(), key=lambda kv: -kv[1]["ms"]):
            extra = f"{d['flops'] / d['ms'] / 1e9:8.1f} TFLOP/s" if d["flops"] else (
                f"{d['bytes'] / d['ms'] / 1e6:8.1f} GB/s" if d["bytes"] else "")
            print(f"  {n:56s} calls {d['calls']:6d}  {d['ms'] / prof_steps:9.2f} ms/step  {100 * d['ms'] / tot:5.1f}%  {extra}",
                  file=sys.stderr)
        print(f"  peak device memory {peak_mem / 2**30:.1f} GiB (whole run); {peak_mem_native / 2**30:.1f} GiB on the product path",
              file=sys.stderr)
        print(f"  sum of kernel time {tot / prof_steps:.1f} ms/step vs profiled step {ms_prof / prof_steps:.1f} ms "
              f"(product path, no events: {ms / args.steps:.1f} ms); model FLOPs/clip "
              f"{(fm['dit'] + fm['enc'] + fm['dec']) / 1e15:.3f} PFLOP", file=sys.stderr)
    if vae_only:
        metric = "VAE decode frames/sec (latent T x 90 x 160 -> 720p)"
        model_flops = fm["dec"]
    else:
        metric = ("upscaled frames/sec SeedVR2-3B 720p->4K" if args.workload == "4k_shard"
                  else f"upscaled frames/sec SeedVR2-{variant.upper()}")
        model_flops = fm["dit"] + fm["enc"] + fm["dec"]
    line = {
        "metric": metric,
        "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": desc, "frames_per_gpu": frames_real, "frames_padded": frames_pad, "resolution": [H, W],
                   "parallelism": f"clip-dp{world}", "color_correction": args.color_correction,
                   "source_resolution": [H // div, W // div], "l2": "inputs/activations per step (>10 GB) exceed L2; no flush needed",
                   "weights": "random init, reference key layout, fp16 checkpoint -> bf16 compute",
                   "model_flops_per_clip": model_flops, "peak_device_memory_gib": round(peak_mem_native / 2**30, 1),
                   "peak_device_memory_whole_run_gib": round(peak_mem / 2**30, 1),
                   "sequencing": "value / e2e: native C++ runtime (svr2_vae_encode, svr2_dit_forward_ws, svr2_vae_decode) in one "
                                 "planned workspace per clip; roofline / kernels: the same kernels launched call by call with CUDA events"},
        "dit_step_ms": dit_step_ms,
        "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": frames_host.numel() * 2,
                "d2h_bytes_per_step": out_host.numel() * 2,
                "launch_mode": graph_note,
                "note": ("SeedVR2Engine.vae_decode on a pinned host latent; decoded frames copied back to host" if vae_only else
                         "SeedVR2Engine.upscale_clip on pinned host frames at the source resolution (resized on the device); result copied back to host")},
        "gpu_launches": launches,
        "roofline": {"bound": "tensor", "kernel": "gemm_tcgen05_kernel (Linear + implicit-GEMM Conv3d + upsample)",
                     "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                     "traffic": traffic, "traffic_detail": traffic_detail, "launches": g_calls, "kernel_ms_per_step": g_ms / prof_steps,
                     "share_of_step": g_ms / ms_prof, "profiled_ms_per_step": ms_prof / prof_steps, "peak_source": peak_src,
                     "note": "achieved = algorithmic FLOPs only (a duplicated QK^T pass of the VAE attention counts as time, not work)"},
        "kernels": kernel_table(prof, prof_steps, peak_tf, peak_gbs, ms_prof / prof_steps),
        "clocks": sampler.result(),
    }
    if args.lib_baseline != "none" and not vae_only:
        lib.release_workspace(dev)       # the library flow allocates through torch: give it the engine's resident block
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import gpu_library_baseline as glb
            gl = {"ops": glb.op_level(dev)}
            if args.lib_baseline in ("default", "full") and variant == "3b":
                gl["phases_cfg2"] = glb.phase_level("cfg2", engine=eng, dev=dev)
            if args.lib_baseline == "full" and variant == "3b":
                gl["phases_4k_shard"] = glb.phase_level("4k_shard", engine=eng, dev=dev)
            line["gpu_library_baseline"] = gl
        except Exception as ex:   # noqa: BLE001 - a reported comparison must not cost the headline line
            line["gpu_library_baseline"] = {"error": f"{type(ex).__name__}: {str(ex)[:300]}"}
    if not args.no_cpu_baseline:
        info = cpu_oracle_sample(frames_pad, H, W)
        line["cpu_baseline"] = {"value": float(f"{frames_real / info['est_clip_seconds']:.2g}"), "unit": "frames/s",
                                "cores": info["cores"], "kind": "port", "extrapolated": True, "sample": info["sample"],
                                "rates_gflops": {k: round(v, 0) for k, v in info["rates_gflops"].items()}}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
