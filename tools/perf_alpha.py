"""RGBA alpha path (csrc/alpha.cu) at the 4K shard (8 frames, 720p alpha -> 2160 x 3840) and BASELINE config 2
(16 frames, 540p alpha -> 1080 x 1920, the decoded sample cropped from 1088): ms per stage and in total, bytes from
the model below, TB/s; beside it the oracle's torch flow on the same GPU and, when cv2 imports, the reference's host
OpenCV edge round trip.  Prints one JSON document; ``--out PATH`` also writes it to PATH (the committed copy is
profiles/alpha_r3.json).

Byte model per output pixel (the sample is bf16 [3,T,H,W] as the VAE decode leaves it; halo re-reads not counted):
  resize   source alpha 2 B per source pixel + resized alpha fp32 4 B
  edges    RGB 6 B twice (flags / maxima, then the map) + edge map 1 B
  refine   stage 1: RGB 6 + resized alpha 4 + (a, b) 8;  stage 2: (a, b) 8 + RGB 6 + edges 1 + bf16 alpha out 2
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from svr2_import import load_package  # noqa: E402

load_package()
from oracle import alpha_oracle  # noqa: E402

lib = importlib.import_module("comfyui_seedvr2_videoupscaler_b200.lib")
alpha_mod = importlib.import_module("comfyui_seedvr2_videoupscaler_b200.alpha")
SHAPES = {"4k_shard": (8, 720, 1280, 2160, 3840), "config2_1080p": (16, 540, 960, 1080, 1920)}
ITERS = 10


def timed(fn, iters=ITERS):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return {"median_ms": round(ts[len(ts) // 2], 4), "min_ms": round(ts[0], 4), "max_ms": round(ts[-1], 4)}


def host_opencv_edges(rgb_n):
    """The reference's detect_edges_batch flow: device -> host copy, OpenCV per frame, back to the device."""
    import cv2
    import numpy as np
    x = rgb_n.float().cpu().numpy()
    if x.min() < 0:
        x = (x + 1) / 2
    x = (x * 255).clip(0, 255).astype(np.uint8)
    out = []
    for t in range(x.shape[0]):
        gray = cv2.cvtColor(x[t].transpose(1, 2, 0), cv2.COLOR_RGB2GRAY)
        gx = cv2.Sobel(gray, cv2.CV_64F, 1, 0, ksize=3)
        gy = cv2.Sobel(gray, cv2.CV_64F, 0, 1, ksize=3)
        e = np.sqrt(gx ** 2 + gy ** 2)
        out.append((e / e.max() * 255).astype(np.uint8))
    return (torch.from_numpy(np.stack(out)).float() / 255.0).unsqueeze(1).to(rgb_n.device)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON document to this path")
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "n/a", "iters": ITERS, "shapes": {}}
    g = torch.Generator(device="cuda").manual_seed(0)
    for name, (T, h, w, H, W) in SHAPES.items():
        yy, xx = torch.meshgrid(torch.linspace(-1, 1, h, device="cuda"), torch.linspace(-1, 1, w, device="cuda"),
                                indexing="ij")
        alpha = ((xx ** 2 + yy ** 2).sqrt() < 0.6).float().expand(T, 1, h, w).bfloat16().contiguous()
        planes = (torch.randn(3, T, H, W, generator=g, device="cuda") * 0.5).clamp(-1, 1).bfloat16()
        sample = planes.permute(1, 0, 2, 3)                 # [T,3,H,W] view, the pipeline's layout
        out = torch.empty(T, H, W, device="cuda", dtype=torch.bfloat16)
        px = T * H * W
        stage_bytes = {"resize": 2.0 * T * h * w + 4.0 * px, "edges": 13.0 * px, "refine": 35.0 * px}
        total_bytes = sum(stage_bytes.values())
        d = {"T": T, "alpha": [h, w], "out": [H, W], "bytes_model_GB": round(total_bytes / 1e9, 3)}
        d["device_path"] = timed(lambda: alpha_mod.upscale_alpha(alpha, None, sample, out=out))
        d["device_path"]["TB_per_s"] = round(total_bytes / d["device_path"]["median_ms"] / 1e9, 2)
        # per stage, one C-ABI call at a time
        need = lib.load().svr2_alpha_scratch_bytes(T, h, w, H, W)
        scratch = torch.empty(need, device="cuda", dtype=torch.uint8)
        up = torch.empty(T, H, W, device="cuda")
        edges = torch.empty(T, H, W, device="cuda", dtype=torch.uint8)
        s = sample.stride()
        calls = {
            "resize": lambda: lib.call("svr2_alpha_resize_f32", lib.ptr(alpha), 1, 0, 0, T, h, w, lib.ptr(up), H, W,
                                       lib.ptr(scratch), need, lib.stream()),
            "edges": lambda: lib.call("svr2_alpha_edges_u8", lib.ptr(sample), 1, s[1], s[0], s[2], T, h, w, H, W,
                                      lib.ptr(edges), lib.ptr(scratch), need, lib.stream()),
            "refine": lambda: lib.call("svr2_alpha_refine", lib.ptr(sample), 1, s[1], s[0], s[2], lib.ptr(up),
                                       lib.ptr(edges), T, h, w, H, W, lib.ptr(out), 1, 1, lib.ptr(scratch), need,
                                       lib.stream()),
        }
        d["stages"] = {}
        for k, fn in calls.items():
            t = timed(fn)
            t["bytes_model_GB"] = round(stage_bytes[k] / 1e9, 3)
            t["TB_per_s"] = round(stage_bytes[k] / t["median_ms"] / 1e9, 2)
            d["stages"][k] = t
        del scratch, up, edges
        d["oracle_torch_flow_same_gpu"] = timed(lambda: alpha_oracle.edge_guided_alpha_upscale(alpha, sample,
                                                                                              resize_on_cpu=False), iters=3)
        try:
            import cv2  # noqa: F401
            rgb_n = (sample.float() + 1) / 2
            d["reference_host_opencv_edges"] = timed(lambda: host_opencv_edges(rgb_n), iters=3)
        except ImportError:
            d["reference_host_opencv_edges"] = "cv2 not importable on this machine: not measured"
        res["shapes"][name] = d
        print(name, json.dumps(d), flush=True)
        del planes, sample, out, alpha
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
