"""TEST INFRASTRUCTURE ONLY — generates tests/golden/alpha_*.npz from the REFERENCE.

Run in the build container (needs the reference tree and OpenCV):

    python -m oracle.make_alpha_golden

It (1) checks the gray formula of ``oracle/alpha_oracle.py`` against OpenCV's ``COLOR_RGB2GRAY`` on all 2^24 RGB
triples, (2) runs the reference's own ``src.core.alpha_upscaling.edge_guided_alpha_upscale`` on CPU fp32 for every case
below, (3) asserts the torch restatement reproduces it bit for bit (edge map, resized alpha, final alpha) and (4) stores
the inputs, the intermediates and the reference output.  The GPU tests compare the CUDA path to these and to the oracle.
"""
from __future__ import annotations

import importlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import alpha_oracle, ref_import  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")

# name: (T, source h, w, upscaled H, W, alpha kind, rgb kind); sizes from resized_size where a case follows the pipeline
ALPHA_CASES = {
    "alpha_binary_img": (1, 24, 32, 48, 64, "binary", "signed"),
    "alpha_gradient_t3": (3, 20, 28, 40, 56, "gradient", "signed"),
    "alpha_const_frame": (2, 16, 24, 32, 48, "binary", "const0"),        # frame 0: constant RGB, edge max 0
    "alpha_below_m1": (2, 16, 20, 32, 40, "binary", "below_m1"),         # min < -1: the edge map normalises twice
    "alpha_nonneg": (2, 18, 18, 36, 36, "gradient", "nonneg"),           # min >= 0: no normalisation
    "alpha_down": (1, 48, 64, 21, 28, "binary", "signed"),               # down-scale: the antialias support widens
    "alpha_odd": (2, 17, 23, 37, 51, "gradient", "signed"),
    # resolution 64, max_resolution 80 on a 30 x 44 clip: the RGB resizes to 64 x 93 then 55 x 80; the alpha goes
    # from 30 x 44 to 55 x 80 in one step
    "alpha_maxres": (1, 30, 44, 55, 80, "binary", "signed"),
}


def alpha_inputs(T, h, w, H, W, akind, rkind, seed=11):
    """Seeded source alpha (T,1,h,w) and decoded-sample RGB (T,3,H,W), both bf16-rounded fp32: a disc per frame whose
    RGB follows the alpha's outline, plus noise."""
    g = torch.Generator().manual_seed(seed)

    def disc(hh, ww, t):
        yy, xx = torch.meshgrid(torch.linspace(-1, 1, hh), torch.linspace(-1, 1, ww), indexing="ij")
        return ((xx - 0.15 * t) ** 2 + (yy + 0.1 * t) ** 2).sqrt()

    alpha, rgb = [], []
    for t in range(T):
        d = disc(h, w, t)
        a = (d < 0.6).float() if akind == "binary" else (1.2 - d).clamp(0, 1) * torch.rand(h, w, generator=g).add(1).div(2)
        alpha.append(a[None])
        D = disc(H, W, t)
        inside = (D < 0.6).float()[None]
        col_in, col_out = torch.rand(3, 1, 1, generator=g) * 2 - 1, torch.rand(3, 1, 1, generator=g) * 2 - 1
        x = inside * col_in + (1 - inside) * col_out + 0.15 * torch.randn(3, H, W, generator=g)
        if rkind == "const0" and t == 0:
            x = torch.full((3, H, W), -0.25)
        elif rkind == "below_m1":
            x = x * 1.6 - 0.2
        elif rkind == "nonneg":
            x = (x + 1) / 2
        rgb.append(x.clamp(-1.6, 1.6) if rkind == "below_m1" else x.clamp(0 if rkind == "nonneg" else -1, 1))
    alpha = torch.stack(alpha).bfloat16().float()
    rgb = torch.stack(rgb).bfloat16().float()
    return alpha, rgb


def run_alpha_cases():
    import cv2

    ref_import.install_stubs()
    ref = importlib.import_module("src.core.alpha_upscaling")
    # the gray formula against OpenCV on all 2^24 RGB triples
    v = np.arange(1 << 24, dtype=np.uint32)
    trip = np.stack([(v >> 16) & 255, (v >> 8) & 255, v & 255], -1).astype(np.uint8).reshape(4096, 4096, 3)
    cvg = cv2.cvtColor(trip, cv2.COLOR_RGB2GRAY)
    t = torch.from_numpy(trip)
    ours = alpha_oracle.gray_u8(t[..., 0], t[..., 1], t[..., 2]).numpy()
    assert np.array_equal(ours, cvg.astype(np.int32)), "gray formula != cv2 COLOR_RGB2GRAY"
    print("alpha: gray == cv2 COLOR_RGB2GRAY on all 2^24 triples")
    for name, (T, h, w, H, W, akind, rkind) in ALPHA_CASES.items():
        alpha, rgb = alpha_inputs(T, h, w, H, W, akind, rkind)
        want = ref.edge_guided_alpha_upscale(alpha.clone(), rgb.clone(), rgb.clone(), method="guided")
        got, inter = alpha_oracle.edge_guided_alpha_upscale(alpha, rgb, intermediates=True)
        rgb_n = (rgb + 1) / 2 if rgb.min() < 0 else rgb
        ref_edges = (ref.detect_edges_batch(rgb_n, method="sobel") * 255.0).round().to(torch.uint8)[:, 0]
        assert torch.equal(inter["edges_u8"], ref_edges), f"{name}: edge map != reference"
        assert torch.equal(alpha_oracle.edge_map(inter["edges_u8"]), ref.detect_edges_batch(rgb_n, method="sobel")), name
        assert torch.equal(got, want), f"{name}: oracle != reference (max {(got - want).abs().max().item():.3g})"
        binary = alpha_oracle.is_binary_mask(alpha)
        norms = int(rgb.min() < 0) + int(rgb_n.min() < 0)
        np.savez_compressed(os.path.join(GOLD, f"{name}.npz"), alpha=alpha.numpy(), rgb=rgb.numpy(),
                            edges_u8=inter["edges_u8"].numpy(), alpha_up=inter["alpha_up"].numpy(), out=want.numpy(),
                            binary=np.bool_(binary), normalisations=np.int32(norms))
        print(f"{name}: T={T} {h}x{w} -> {H}x{W} binary={binary} normalisations={norms}  oracle == reference")


def main():
    os.makedirs(GOLD, exist_ok=True)
    run_alpha_cases()


if __name__ == "__main__":
    main()
