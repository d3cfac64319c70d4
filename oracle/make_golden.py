"""TEST INFRASTRUCTURE ONLY — generates tests/golden/*.npz from the REFERENCE.

Run in the build container (needs /root/reference):

    python -m oracle.make_golden

For each case it (1) builds the reference's own module (NaDiT 3B/7B structure at
reduced width, full-width VideoAutoencoderKLWrapper) through
``oracle/ref_import.py``, (2) loads the deterministic synthetic checkpoint from
``comfyui-seedvr2_videoupscaler_b200/weights.py``, (3) runs the reference forward on CPU fp32
on seeded inputs, (4) asserts the restatements in ``oracle/dit_oracle.py`` /
``oracle/vae_oracle.py`` reproduce it, and (5) stores the reference outputs.
The fixtures pin the oracle; the GPU tests compare the CUDA path to the oracle.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import dit_oracle, dropin, vae_oracle  # noqa: E402
from oracle import ref_import  # noqa: E402
from oracle.ref_import import import_reference_dit, import_reference_vae  # noqa: E402
from svr2_import import load_package  # noqa: E402

pkg = load_package()
GOLD = os.path.join(ROOT, "tests", "golden")

DIT_CASES = {
    # name: (variant, cfg overrides, (T, H, W) latent, txt_len)
    "dit3b_tiny_t3": ("3b", dict(dim=256, heads=2, layers=4, mm_layers=2, txt_in_dim=64), (3, 40, 72), 58),
    "dit3b_tiny_t5": ("3b", dict(dim=256, heads=2, layers=4, mm_layers=2, txt_in_dim=64), (5, 16, 24), 58),
    "dit3b_tiny_img": ("3b", dict(dim=256, heads=2, layers=2, mm_layers=1, txt_in_dim=64), (1, 64, 64), 58),
    "dit7b_tiny_t3": ("7b", dict(dim=384, heads=3, layers=3, mm_layers=3, txt_in_dim=64), (3, 40, 72), 58),
}


def dit_inputs(cfg, T, H, W, l, seed=42):
    g = torch.Generator().manual_seed(seed)
    vid = torch.randn(T * H * W, cfg["in_ch"], generator=g)
    txt = torch.randn(l, cfg["txt_in_dim"], generator=g)
    return vid, txt


def build_ref_dit(cfg):
    variant = cfg["variant"]
    mod = import_reference_dit(variant)
    L = cfg["layers"]
    common = dict(vid_in_channels=cfg["in_ch"], vid_out_channels=cfg["out_ch"], vid_dim=cfg["dim"],
                  txt_in_dim=cfg["txt_in_dim"], txt_dim=cfg["dim"], emb_dim=6 * cfg["dim"],
                  heads=cfg["heads"], head_dim=cfg["head_dim"], expand_ratio=4, norm="fusedrms",
                  norm_eps=1e-5, ada="single", qk_bias=False, qk_norm="fusedrms", patch_size=[1, 2, 2],
                  num_layers=L, block_type=L * ["mmdit_sr"], window=L * [(4, 3, 3)],
                  window_method=[("720pwin_by_size_bysize", "720pswin_by_size_bysize")[i % 2] for i in range(L)])
    if variant == "3b":
        net = mod.NaDiT(vid_out_norm="fusedrms", txt_in_norm="fusedln", mm_layers=cfg["mm_layers"],
                        mlp_type="swiglu", msa_type=None, rope_type="mmrope3d", rope_dim=128, **common)
    else:
        net = mod.NaDiT(qk_rope=True, shared_mlp=False, shared_qkv=False, mlp_type="normal", **common)
    return net.eval()


def run_dit_case(name):
    variant, over, (T, H, W), l = DIT_CASES[name]
    cfg = dit_oracle.dit_config(variant, **over)
    sd = pkg.weights.synth_dit_state_dict(cfg, seed=1234, dtype=torch.float16)
    sd32 = {k: v.float() for k, v in sd.items()}
    net = build_ref_dit(cfg)
    missing = net.load_state_dict(sd32, strict=True)
    vid, txt = dit_inputs(cfg, T, H, W, l)
    with torch.no_grad():
        kw = {} if variant == "3b" else {}
        ref = net(vid=vid.clone(), txt=txt.clone(), vid_shape=torch.tensor([[T, H, W]]),
                  txt_shape=torch.tensor([[l]]), timestep=torch.tensor([1000.0]), **kw).vid_sample
    taps = {}
    ora = dit_oracle.dit_forward(sd32, cfg, vid, txt, T, H, W, mode="fp32", taps=taps)
    err = (ora - ref).abs().max().item()
    scale = ref.abs().max().item()
    print(f"[{name}] ref |max|={scale:.3f} rms={ref.pow(2).mean().sqrt():.3f} oracle-vs-reference max|d|={err:.2e}")
    assert err < 2e-4 * max(scale, 1.0), f"{name}: oracle deviates from reference ({err})"
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), out=ref.numpy().astype(np.float32),
                        meta=np.array([T, H, W, l]),
                        emb=taps["emb"].numpy(), block0=taps["block0"][::37].numpy())


VAE_CASES = {
    "vae_dec_t3": ("decode", (3, 4, 6)),     # latent T,h,w -> 9 frames 32x48
    "vae_dec_img": ("decode", (1, 6, 4)),
    "vae_enc_t9": ("encode", (9, 32, 48)),   # frames T,H,W -> latent 3x4x6
    "vae_enc_img": ("encode", (1, 48, 32)),
}


def build_ref_vae():
    mod = import_reference_vae()
    vae = mod.VideoAutoencoderKLWrapper(
        act_fn="silu", block_out_channels=[128, 256, 512, 512], down_block_types=["DownEncoderBlock3D"] * 4,
        in_channels=3, latent_channels=16, layers_per_block=2, norm_num_groups=32, out_channels=3,
        slicing_sample_min_size=4, temporal_scale_num=2, inflation_mode="pad",
        up_block_types=["UpDecoderBlock3D"] * 4, spatial_downsample_factor=8, temporal_downsample_factor=4,
        use_quant_conv=False, use_post_quant_conv=False, freeze_encoder=False)
    return vae.eval()


def run_vae_cases():
    sd = pkg.weights.synth_vae_state_dict(seed=4321, dtype=torch.float16)
    sd32 = {k: v.float() for k, v in sd.items()}
    vae = build_ref_vae()
    res = vae.load_state_dict(dict(sd32), strict=True)
    print("vae load:", res)
    # the reference pipeline enables temporal slicing (model_configuration.py:1247-1259)
    vae.set_causal_slicing(split_size=4, memory_device="same")
    for name, (kind, shp) in VAE_CASES.items():
        g = torch.Generator().manual_seed(7)
        if kind == "decode":
            T, h, w = shp
            z = torch.randn(1, 16, T, h, w, generator=g)
            with torch.no_grad():
                ref = vae.decode(z).sample
                if ref.ndim == 4:
                    ref = ref.unsqueeze(2)
            ora = vae_oracle.vae_decode(sd32, z)
        else:
            T, H, W = shp
            x = torch.rand(1, 3, T, H, W, generator=g) * 2 - 1
            with torch.no_grad():
                ref = vae.encode(x).latent
                if ref.ndim == 4:
                    ref = ref.unsqueeze(2)
            ora = vae_oracle.vae_encode(sd32, x)
        err = (ora - ref).abs().max().item()
        scale = ref.abs().max().item()
        print(f"[{name}] out {tuple(ref.shape)} |max|={scale:.3f} oracle-vs-reference max|d|={err:.2e}")
        assert err < 2e-4 * max(scale, 1.0), name
        np.savez_compressed(os.path.join(GOLD, name + ".npz"), out=ref.numpy().astype(np.float32),
                            meta=np.array(shp))


# ---- spatially tiled VAE (attn_video_vae.py:1302-1630): name -> (kind, shape, tile_size, tile_overlap)
TILED_CASES = {
    "vae_tiled_dec_t2": ("decode", (2, 7, 11), (32, 32), (16, 16)),     # latent 7x11, tiles of 4 with 2 overlap, ragged edge
    "vae_tiled_enc_t5": ("encode", (5, 56, 88), (32, 32), (16, 16)),
    "vae_tiled_dec_img": ("decode", (1, 9, 6), (48, 32), (8, 24)),      # single image, anisotropic tiles / overlaps
}


def run_tiled_cases():
    sd = pkg.weights.synth_vae_state_dict(seed=4321, dtype=torch.float16)
    sd32 = {k: v.float() for k, v in sd.items()}
    vae = build_ref_vae()
    vae.load_state_dict(dict(sd32), strict=True)
    vae.set_causal_slicing(split_size=4, memory_device="same")
    vae.debug, vae.tensor_offload_device = None, None          # set by apply_model_specific_config in the pipeline
    for name, (kind, shp, tile, ov) in TILED_CASES.items():
        g = torch.Generator().manual_seed(7)
        with torch.no_grad():
            if kind == "decode":
                z = torch.randn(1, 16, *shp, generator=g)
                ref = vae.decode(z, tiled=True, tile_size=tile, tile_overlap=ov).sample
                ora = vae_oracle.tiled_decode(sd32, z, tile, ov)
            else:
                x = torch.rand(1, 3, *shp, generator=g) * 2 - 1
                ref = vae.encode(x, tiled=True, tile_size=tile, tile_overlap=ov).latent
                ora = vae_oracle.tiled_encode(sd32, x, tile, ov)
        if ref.ndim == 4:
            ref = ref.unsqueeze(2)
        if ora.ndim == 4:
            ora = ora.unsqueeze(2)
        err = (ora - ref).abs().max().item()
        print(f"[{name}] out {tuple(ref.shape)} oracle-vs-reference max|d|={err:.2e}")
        assert err < 2e-4 * max(ref.abs().max().item(), 1.0), name
        np.savez_compressed(os.path.join(GOLD, name + ".npz"), out=ref.numpy().astype(np.float32),
                            meta=np.array(list(shp) + list(tile) + list(ov)))


# ---- post-decode colour correction (src/utils/color_fix.py): name -> (T, H, W)
COLOR_CASES = {
    "color_t2_40x56": (2, 40, 56),        # min(H,W)//8 = 5 caps the dilation of levels 3, 4
    "color_t1_72x96": (1, 72, 96),
    "color_t3_130x150": (3, 130, 150),    # all five dilations (1..16) un-capped, odd width
}
COLOR_METHODS = ("wavelet", "adain", "lab")


def color_inputs(T, H, W, seed=7):
    """(content, style) bf16 [T,3,H,W] in [-1,1]: a smooth scene plus detail (content) / a colour-shifted,
    softer version of it (style) — what the decoder output and the resized input clip look like."""
    g = torch.Generator().manual_seed(seed)
    base = torch.nn.functional.interpolate(torch.randn(T, 3, H // 8 + 1, W // 8 + 1, generator=g), size=(H, W),
                                           mode="bilinear", align_corners=False)
    content = (base + 0.15 * torch.randn(T, 3, H, W, generator=g)).clamp(-1, 1).to(torch.bfloat16)
    style = (0.8 * base + 0.1 + 0.05 * torch.randn(T, 3, H, W, generator=g)).clamp(-1, 1).to(torch.bfloat16)
    return content, style


def run_color_cases():
    """Reference outputs of src/utils/color_fix.py on CPU bf16 inputs; the oracle must reproduce wavelet / AdaIN
    bit for bit and LAB up to the tie order of the reference's unstable sort."""
    import importlib
    if ref_import.REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, ref_import.REFERENCE_ROOT)
    ref = importlib.import_module("src.utils.color_fix")
    from oracle import color_oracle as co

    class _Dbg:
        def log(self, *a, **k):
            pass

    for name, (T, H, W) in COLOR_CASES.items():
        content, style = color_inputs(T, H, W)
        outs = {
            "wavelet": ref.wavelet_reconstruction(content.clone(), style.clone(), _Dbg()),
            "adain": ref.adaptive_instance_normalization(content.clone(), style.clone()),
            "lab": ref.lab_color_transfer(content.clone(), style.clone(), _Dbg(), luminance_weight=0.8),
        }
        assert all(v.dtype == torch.bfloat16 for v in outs.values())
        assert torch.equal(outs["wavelet"].float(), co.wavelet_reconstruction(content, style)), name
        assert torch.equal(outs["adain"].float(), co.adaptive_instance_normalization(content, style)), name
        lab_o = co.lab_color_transfer(content, style)
        same = (outs["lab"].float() == lab_o).float().mean().item()
        mse = ((outs["lab"].float() - lab_o) ** 2).mean().item()
        psnr = 99.0 if mse == 0 else 10 * np.log10(4.0 / mse)
        assert same > 0.99 and psnr > 60.0, (name, same, psnr)
        print(f"{name}: wavelet/adain oracle == reference (bit-exact); lab {100 * same:.2f}% equal, {psnr:.1f} dB")
        if name == "color_t2_40x56":
            # hsv / wavelet_adaptive (not shipped by the engine yet): saturation has heavy ties (a third of the values),
            # so the reference's unstable sort leaves the result defined only up to the tie order — pin the colour-space
            # conversions bit for bit and the result as a distribution.
            tint = torch.tensor([1.0, 0.6, 0.3]).view(1, 3, 1, 1)
            c2, s2 = (content.float() * tint).to(torch.bfloat16), (style.float() * tint * 0.9).to(torch.bfloat16)
            c01 = ((c2.float() + 1.0) * 0.5).clamp(0.0, 1.0)
            assert torch.equal(ref._rgb_to_hsv_batch(c01.clone()), co.rgb_to_hsv(c01))
            assert torch.equal(ref._hsv_to_rgb_batch(co.rgb_to_hsv(c01)), co.hsv_to_rgb(co.rgb_to_hsv(c01)))
            outs["hsv"] = ref.hsv_saturation_histogram_match(c2.clone(), s2.clone(), _Dbg())
            outs["wavelet_adaptive"] = ref.wavelet_adaptive_color_correction(c2.clone(), s2.clone(), _Dbg())
            for key, fn in (("hsv", co.hsv_saturation_histogram_match), ("wavelet_adaptive", co.wavelet_adaptive_color_correction)):
                o = fn(c2, s2)
                sat = lambda x: co.saturation_map(x.float()).flatten().sort().values
                dsat = (sat(o) - sat(outs[key])).abs()
                db = 10 * np.log10(4.0 / ((o - outs[key].float()) ** 2).mean().item())
                print(f"   {key}: sorted-saturation diff max {dsat.max().item():.4f} mean {dsat.mean().item():.5f}, {db:.1f} dB")
                assert dsat.mean() < 2e-3 and db > 35.0, key
            print(f"{name}: hsv / wavelet_adaptive oracle == reference as distributions (tie order is unspecified)")
        np.savez_compressed(os.path.join(GOLD, name + ".npz"),
                            **{k: v.float().numpy().astype(np.float32) for k, v in outs.items()})
    # temporal-overlap cross-fade (src/core/generation_utils.py:284-312), bit for bit for every overlap length
    gu_src = open(os.path.join(ref_import.REFERENCE_ROOT, "src/core/generation_utils.py")).read()
    start = gu_src.index("def blend_overlapping_frames")
    ns = {"torch": torch}
    exec(gu_src[start:gu_src.index("\ndef ", start + 10)], ns)     # the function only (its module needs a GPU stack)
    g = torch.Generator().manual_seed(21)
    blends = {}
    for ov in (1, 2, 3, 4, 7, 8):
        a = torch.rand(ov, 6, 8, 3, generator=g).to(torch.bfloat16)
        b = torch.rand(ov, 6, 8, 3, generator=g).to(torch.bfloat16)
        ref_out = ns["blend_overlapping_frames"](a, b, ov)
        assert ref_out.dtype == torch.bfloat16
        assert torch.equal(ref_out.float(), co.blend_overlapping_frames(a, b, ov)), ov
        blends[f"ov{ov}"] = ref_out.float().numpy().astype(np.float32)
    for ov in (2, 5):       # fp32 frames: the multi-GPU merge of inference_cli.py:1241-1270
        a, b = torch.rand(ov, 6, 8, 3, generator=g), torch.rand(ov, 6, 8, 3, generator=g)
        ref_out = ns["blend_overlapping_frames"](a, b, ov)
        assert ref_out.dtype == torch.float32 and torch.equal(ref_out, co.blend_overlapping_frames(a, b, ov)), ov
        blends[f"f32_ov{ov}"] = ref_out.numpy()
    print("blend_overlapping_frames: oracle == reference (bit-exact) for overlaps 1,2,3,4,7,8 (bf16) and 2,5 (fp32)")
    # temporal padding with reversed frames (src/core/generation_utils.py:598-657): frame-index sequences
    start = gu_src.index("def pad_video_temporal")
    exec(gu_src[start:gu_src.index("\ndef ", start + 10)], ns)
    ns.setdefault("Optional", __import__("typing").Optional)
    pads = {}
    for t in range(1, 14):
        idx = torch.arange(t, dtype=torch.float32).view(1, t, 1, 1)                 # c t h w, value = frame index
        auto = ns["pad_video_temporal"](idx, temporal_dim=1)
        assert torch.equal(auto, vae_oracle.pad_video_temporal(idx, temporal_dim=1)), t
        pads[f"auto_t{t}"] = auto.flatten().numpy()
        for count in (1, 3, t, t + 2):
            for prepend in (False, True):
                r = ns["pad_video_temporal"](idx, count=count, temporal_dim=1, prepend=prepend)
                assert torch.equal(r, vae_oracle.pad_video_temporal(idx, count, 1, prepend)), (t, count, prepend)
                pads[f"t{t}_c{count}_{'pre' if prepend else 'app'}"] = r.flatten().numpy()
    print("pad_video_temporal: oracle == reference for t = 1..13, explicit counts, append / prepend")
    np.savez_compressed(os.path.join(GOLD, "pad_temporal.npz"), **pads)
    np.savez_compressed(os.path.join(GOLD, "blend_overlap.npz"), **blends)


# ---- clip pre-processing (prepare_video_transforms): name -> (T, h, w, resolution, max_resolution)
PRE_CASES = {
    "pre_up3x": (2, 30, 41, 90, 0),              # 3x up-scale, odd sizes, pad 90x123 -> 96x128
    "pre_up_landscape": (1, 45, 80, 72, 0),
    "pre_down": (2, 64, 48, 40, 0),              # down-scale: the antialias support widens
    "pre_capped": (1, 36, 64, 108, 160),         # max_resolution triggers the second resize
    "pre_identity": (2, 33, 57, 33, 0),          # already at the target size
}


def pre_inputs(T, h, w, seed=3):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(T, h, w, 3, generator=g) * 1.1 - 0.05     # [T,h,w,3], slightly outside [0,1]


def run_pre_cases():
    """The reference's own transform classes composed as prepare_video_transforms does
    (src/core/generation_utils.py:72-84), run on CPU on the bf16 clip (generation_phases.py:380-413)."""
    import importlib
    if ref_import.REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, ref_import.REFERENCE_ROOT)
    na = importlib.import_module("src.data.image.transforms.na_resize")
    dc = importlib.import_module("src.data.image.transforms.divisible_crop")
    from torchvision.transforms import Compose, Lambda, Normalize
    from oracle import pre_oracle

    for name, (T, h, w, res, mx) in PRE_CASES.items():
        tf = Compose([na.NaResize(resolution=res, mode="side", downsample_only=False, max_resolution=mx),
                      Lambda(lambda x: torch.clamp(x, 0.0, 1.0)), dc.DivisiblePad((16, 16)), Normalize(0.5, 0.5),
                      Lambda(lambda x: x.permute(1, 0, 2, 3))])
        frames = pre_inputs(T, h, w)
        ref = tf(frames.to(torch.bfloat16).permute(0, 3, 1, 2))
        assert ref.dtype == torch.bfloat16
        ora = pre_oracle.preprocess(frames, res, mx)
        d = (ref.float() - ora).abs()
        same = (d == 0).float().mean().item()
        assert ref.shape == ora.shape and same > 0.999 and d.max().item() <= 2 ** -7, (name, same, d.max().item())
        print(f"{name}: {tuple(ref.shape)} oracle vs reference transform {100 * same:.3f}% bit-equal, max {d.max().item():.4f}")
        np.savez_compressed(os.path.join(GOLD, name + ".npz"), out=ref.float().numpy().astype(np.float32))


def main():
    os.makedirs(GOLD, exist_ok=True)
    torch.manual_seed(0)
    if "--tiled-only" in sys.argv:
        return run_tiled_cases()
    if "--dropin-only" in sys.argv:
        return dropin.record_reference(pkg, os.path.join(GOLD, "dropin_runner.npz"))
    if "--color-only" not in sys.argv and "--pre-only" not in sys.argv:
        for name in DIT_CASES:
            run_dit_case(name)
        run_vae_cases()
        run_tiled_cases()
        dropin.record_reference(pkg, os.path.join(GOLD, "dropin_runner.npz"))
    if "--pre-only" not in sys.argv:
        run_color_cases()
    if "--color-only" not in sys.argv:
        run_pre_cases()


if __name__ == "__main__":
    main()
