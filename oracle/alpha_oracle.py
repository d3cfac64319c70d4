"""TEST INFRASTRUCTURE ONLY — never imported by the product path.

Torch restatement of the reference's edge-guided alpha upscaling (``edge_guided_alpha_upscale``,
``src/core/alpha_upscaling.py:289-438``) without OpenCV, so that it runs on the GPU next to the CUDA path.

Third-party algorithms restated (``detect_edges_batch``, ``alpha_upscaling.py:141-186``):
- OpenCV 4.13 ``cvtColor(COLOR_RGB2GRAY)`` on 8-bit input: ``(9798 R + 19235 G + 3735 B + 16384) >> 15``;
- ``cv2.Sobel(gray, CV_64F, dx, dy, ksize=3)`` with the default ``BORDER_REFLECT_101``;
- NumPy's ``(x * 255).clip(0, 255).astype(uint8)`` and ``(edge / edge.max() * 255).astype(uint8)`` in fp64, whose
  0/0 on a frame without edges casts to 0.
The edge map goes back to torch as ``u8.float() / 255.0`` computed on the CPU (a true division; torch's CUDA division
by a scalar multiplies by the reciprocal, which differs in the last bit for some bytes), here as a 256-entry table.
The alpha resize runs on the CPU by default: the CUDA kernel's tap tables (``csrc/pre.cu``) follow torch's CPU weight
computation, which differs from torch's CUDA one in the last bits (up to ~2e-6 on the resized alpha).
Everything after the edge map is the reference's own torch code.  Pinned: ``python -m oracle.make_alpha_golden``
asserts this restatement equals the reference bit for bit (``tests/golden/alpha_*.npz``) and the gray formula equals
``cv2`` on all 2^24 RGB triples.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

_EDGE_LUT = torch.arange(256, dtype=torch.float32) / 255.0      # on the CPU, as the reference divides


def gray_u8(r: torch.Tensor, g: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """cv2 COLOR_RGB2GRAY of 8-bit channels (any integer dtype) -> int32."""
    return (9798 * r.int() + 19235 * g.int() + 3735 * b.int() + 16384) >> 15


def _reflect101(n: int, device) -> torch.Tensor:
    """Source index of positions -1 .. n under BORDER_REFLECT_101."""
    i = torch.arange(-1, n + 1, device=device).abs()
    i = torch.where(i >= n, 2 * n - 2 - i, i)
    return i.clamp(0, n - 1)


def sobel_edges_u8(images: torch.Tensor) -> torch.Tensor:
    """detect_edges_batch(images, 'sobel') before the final / 255: (T, 3, H, W) float -> (T, H, W) uint8."""
    x = images.float()
    if x.min() < 0:
        x = (x + 1) / 2
    u8 = (x * 255).clamp(0, 255).to(torch.uint8)
    gray = gray_u8(u8[:, 0], u8[:, 1], u8[:, 2])
    T, H, W = gray.shape
    p = gray.index_select(1, _reflect101(H, gray.device)).index_select(2, _reflect101(W, gray.device)).long()
    c = lambda dy, dx: p[:, 1 + dy:1 + dy + H, 1 + dx:1 + dx + W]      # noqa: E731
    gx = (c(-1, 1) - c(-1, -1)) + 2 * (c(0, 1) - c(0, -1)) + (c(1, 1) - c(1, -1))
    gy = (c(1, -1) - c(-1, -1)) + 2 * (c(1, 0) - c(-1, 0)) + (c(1, 1) - c(-1, 1))
    mag = torch.sqrt((gx * gx + gy * gy).double())
    mx = mag.flatten(1).max(1).values.view(T, 1, 1)
    e = torch.where(mx > 0, mag / mx * 255, torch.zeros_like(mag))
    return e.to(torch.uint8)


def edge_map(edges_u8: torch.Tensor) -> torch.Tensor:
    """(T, H, W) uint8 -> (T, 1, H, W) fp32 in [0, 1], bit-equal to the reference's CPU division."""
    return _EDGE_LUT.to(edges_u8.device)[edges_u8.long()].unsqueeze(1)


def _box(x: torch.Tensor, r: int) -> torch.Tensor:
    return F.avg_pool2d(x, kernel_size=2 * r + 1, stride=1, padding=r)


def guided_filter(guide: torch.Tensor, src: torch.Tensor, radius: int, eps: float) -> torch.Tensor:
    """guided_filter_pytorch + _apply_guided_filter (alpha_upscaling.py:189-286)."""
    I = guide.mean(dim=1, keepdim=True) if guide.shape[1] == 3 else guide
    mean_I, mean_p = _box(I, radius), _box(src, radius)
    corr_I, corr_Ip = _box(I * I, radius), _box(I * src, radius)
    var_I = corr_I - mean_I * mean_I
    cov_Ip = corr_Ip - mean_I * mean_p
    a = cov_Ip / (var_I + eps)
    b = mean_p - a * mean_I
    return _box(a, radius) * I + _box(b, radius)


def is_binary_mask(alpha: torch.Tensor) -> bool:
    flat = alpha.float().flatten()
    ratio = ((flat < 0.1).sum().float() + (flat > 0.9).sum().float()) / flat.numel()
    return bool(ratio > 0.95)


def edge_guided_alpha_upscale(input_alpha: torch.Tensor, upscaled_rgb: torch.Tensor, intermediates: bool = False,
                              resize_on_cpu: bool = True):
    """input_alpha (T, 1, h, w), upscaled_rgb (T, 3, H, W) -> fp32 (T, 1, H, W) in [0, 1].  With ``intermediates``
    also returns a dict of the edge map (uint8), the resized alpha, the guided-filter output ``q`` and the alpha before
    the final snap (``mid``, binary masks only)."""
    T, _, H, W = upscaled_rgb.shape
    alpha = input_alpha.float()
    rgb = upscaled_rgb.float()
    binary = is_binary_mask(alpha)
    rgb_n = (rgb + 1) / 2 if rgb.min() < 0 else rgb
    edges_u8 = sobel_edges_u8(rgb_n)
    edge = edge_map(edges_u8)
    up = F.interpolate(alpha.cpu() if resize_on_cpu else alpha, size=(H, W), mode="bicubic", align_corners=False,
                       antialias=True).clamp(0, 1).to(alpha.device)
    inter = {"edges_u8": edges_u8, "alpha_up": up}
    if binary:
        q = guided_filter(rgb_n, up, radius=2, eps=0.002)
        transition = F.max_pool2d(edge, kernel_size=3, stride=1, padding=1)
        is_solid = transition < 0.05
        alpha_binary = (q > 0.5).float()
        contrast = torch.sigmoid((q - 0.5) * 12.0)
        strength = torch.clamp(edge / 0.25, 0, 1)
        alpha_in_edges = q * (1 - strength) + contrast * strength
        combined = torch.where(is_solid, alpha_binary, alpha_in_edges)
        final = torch.where(transition < 0.03, (combined > 0.5).float(), combined)
        should_be_binary = (final > 0.3) & (final < 0.7) & ~(edge > 0.15)
        inter["mid"] = final
        final = torch.where(should_be_binary, (final > 0.5).float(), final)
    else:
        q = guided_filter(rgb_n, up, radius=3, eps=0.002)
        final = q
    inter["q"] = q
    final = final.clamp(0, 1)
    return (final, inter) if intermediates else final
