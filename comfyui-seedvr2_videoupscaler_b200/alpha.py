"""Alpha channel of RGBA clips: edge-guided upscaling on the device (``csrc/alpha.cu``).

Mirrors ``src/core/alpha_upscaling.py`` of the reference: the source alpha is resized (antialiased bicubic) straight
to the output size, then a guided filter steered by the upscaled RGB sharpens it, with an extra edge-aware refinement
for binary masks.  The reference's edge map copies the clip to the host and runs OpenCV frame by frame; here it is an
integer-exact CUDA kernel, and the three data-dependent decisions (binary mask; normalising the RGB once or twice)
stay on the device, so the whole path captures into a CUDA graph.  GPU only: there is no CPU fallback.
"""
from __future__ import annotations

from typing import List, Optional

import torch

from . import lib

_IN_DTYPES = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}
_RGB_DTYPES = {torch.float32: 0, torch.bfloat16: 1}
_OUT_DTYPES = {torch.float32: 0, torch.bfloat16: 1}


def upscale_alpha(alpha: torch.Tensor, channel: Optional[int], sample: torch.Tensor,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Edge-guided upscale of a source alpha to the size of ``sample``.

    ``alpha``: ``[T, h, w, C]`` with the alpha at ``channel`` (ComfyUI / CLI frames), or ``[T, 1, h, w]`` with
    ``channel=None``; fp32, bf16 or fp16, rounded to bf16 on load.  ``sample``: the decoded ``[T, 3, H, W]`` RGB before
    colour correction, fp32 or bf16, any strides with contiguous pixels (e.g. a permuted view of the VAE output).
    ``out``: ``[T, 1, H, W]`` (default, fp32) or a ``[T, H, W]`` view with pixel stride 1 or 4 (the alpha slot of a
    ``[T, H, W, 4]`` image), fp32 or bf16.  Returns ``out``."""
    if not (alpha.is_cuda and sample.is_cuda):
        raise lib.Svr2Error("alpha upscaling runs on the GPU only (no CPU fallback)")
    if sample.ndim != 4 or sample.shape[1] != 3:
        raise ValueError(f"sample must be [T, 3, H, W], got {tuple(sample.shape)}")
    if alpha.ndim != 4 or (channel is None and alpha.shape[1] != 1):
        raise ValueError(f"alpha must be [T, 1, h, w] or [T, h, w, C] with a channel, got {tuple(alpha.shape)}")
    T, _, H, W = sample.shape
    if alpha.shape[0] != T:
        raise ValueError(f"alpha has {alpha.shape[0]} frames, the RGB {T}")
    if alpha.dtype not in _IN_DTYPES:
        alpha = alpha.float()
    alpha = alpha.contiguous()
    if channel is None:
        h, w, C, ch = alpha.shape[2], alpha.shape[3], 0, 0
    else:
        h, w, C, ch = alpha.shape[1], alpha.shape[2], alpha.shape[3], int(channel)
        if not 0 <= ch < C:
            raise ValueError(f"alpha channel {ch} outside [0, {C})")
    if sample.dtype not in _RGB_DTYPES:
        sample = sample.float()
    if sample.stride(3) != 1:
        sample = sample.contiguous()
    if out is None:
        out = torch.empty(T, 1, H, W, device=sample.device, dtype=torch.float32)
    if out.dtype not in _OUT_DTYPES or out.numel() != T * H * W:
        raise ValueError(f"out must hold T*H*W fp32 or bf16 values, got {tuple(out.shape)} {out.dtype}")
    ostride = out.stride(-1)
    if tuple(out.stride()) not in ((H * W, H * W, W, 1), (H * W * ostride, W * ostride, ostride)):
        raise ValueError(f"out must be [T, 1, H, W] contiguous or a [T, H, W] view with a pixel stride, got strides "
                         f"{tuple(out.stride())}")
    dev = sample.device
    need = lib.load().svr2_alpha_scratch_bytes(T, h, w, H, W)
    scratch = torch.empty(need, device=dev, dtype=torch.uint8)
    up = torch.empty(T, H, W, device=dev, dtype=torch.float32)
    edges = torch.empty(T, H, W, device=dev, dtype=torch.uint8)
    cs, ts, rs = sample.stride(1), sample.stride(0), sample.stride(2)
    rgb_dt, px = _RGB_DTYPES[sample.dtype], T * H * W
    lib.call("svr2_alpha_resize_f32", lib.ptr(alpha), _IN_DTYPES[alpha.dtype], C, ch, T, h, w, lib.ptr(up), H, W,
             lib.ptr(scratch), need, lib.stream(), nbytes=alpha.numel() / max(C, 1) * alpha.element_size() + 4.0 * px)
    lib.call("svr2_alpha_edges_u8", lib.ptr(sample), rgb_dt, cs, ts, rs, T, h, w, H, W, lib.ptr(edges),
             lib.ptr(scratch), need, lib.stream(), nbytes=2 * 3.0 * px * sample.element_size() + px)
    lib.call("svr2_alpha_refine", lib.ptr(sample), rgb_dt, cs, ts, rs, lib.ptr(up), lib.ptr(edges), T, h, w, H, W,
             lib.ptr(out), _OUT_DTYPES[out.dtype], ostride, lib.ptr(scratch), need, lib.stream(),
             nbytes=px * (2 * 3.0 * sample.element_size() + 4 + 8 + 8 + 1 + out.element_size()))
    return out


def edge_guided_alpha_upscale(input_alpha: torch.Tensor, input_rgb: Optional[torch.Tensor], upscaled_rgb: torch.Tensor,
                              method: str = "guided", debug=None) -> torch.Tensor:
    """``alpha_upscaling.edge_guided_alpha_upscale``: input_alpha ``[T, 1, h, w]`` in [0, 1], upscaled_rgb
    ``[T, 3, H, W]`` in [-1, 1] or [0, 1] -> fp32 ``[T, 1, H, W]`` in [0, 1].  Like the reference, ``input_rgb`` and
    ``method`` are not used.  Frame counts that differ raise ``ValueError`` (the reference fails to broadcast)."""
    return upscale_alpha(input_alpha, None, upscaled_rgb)


def process_alpha_for_batch(rgb_samples: List[torch.Tensor], alpha_original: torch.Tensor, rgb_original: torch.Tensor,
                            device, compute_dtype: torch.dtype, debug=None) -> List[torch.Tensor]:
    """``alpha_upscaling.process_alpha_for_batch``: every sample ``[T, C, H, W]`` (or ``[C, H, W]``) becomes
    ``[T, 4, H, W]`` (``[4, H, W]``) in ``compute_dtype`` = its RGB + the alpha upscaled against it."""
    device = torch.device(device)
    alpha4 = alpha_original.to(device)
    if alpha4.ndim == 3:
        alpha4 = alpha4.unsqueeze(1)
    out = []
    for s in rgb_samples:
        s = s.to(device)
        single = s.ndim == 3
        s4 = s.unsqueeze(0) if single else s
        a = edge_guided_alpha_upscale(alpha4[:, :1], None, s4[:, :3]).to(compute_dtype)
        rgba = torch.cat([s4[:, :3].to(compute_dtype), a], 1)
        out.append(rgba.squeeze(0) if single else rgba)
    return out
