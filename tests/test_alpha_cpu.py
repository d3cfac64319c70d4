"""RGBA alpha upscaling on the CPU: the torch oracle against the reference's goldens, and the ``keep_alpha`` control flow
of the clip runner with the GPU stages stubbed (the kernels are covered by tests/test_alpha_gpu.py)."""
import glob
import importlib
import os

import numpy as np
import pytest
import torch

from oracle import alpha_oracle

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ALPHA_GOLDENS = sorted(glob.glob(os.path.join(GOLD, "alpha_*.npz")))


def test_alpha_goldens_cover_every_decision():
    assert len(ALPHA_GOLDENS) >= 8
    seen = {(bool(d["binary"]), int(d["normalisations"])) for d in map(np.load, ALPHA_GOLDENS)}
    assert {b for b, _ in seen} == {True, False} and {n for _, n in seen} == {0, 1, 2}


@pytest.mark.parametrize("path", ALPHA_GOLDENS, ids=lambda p: os.path.basename(p)[:-4])
def test_alpha_oracle_reproduces_golden(path):
    d = np.load(path)
    alpha, rgb = torch.from_numpy(d["alpha"]), torch.from_numpy(d["rgb"])
    out, inter = alpha_oracle.edge_guided_alpha_upscale(alpha, rgb, intermediates=True)
    assert torch.equal(inter["edges_u8"], torch.from_numpy(d["edges_u8"]))
    assert torch.equal(inter["alpha_up"], torch.from_numpy(d["alpha_up"]))
    assert torch.equal(out, torch.from_numpy(d["out"]))
    assert alpha_oracle.is_binary_mask(alpha) == bool(d["binary"])


def test_alpha_oracle_edge_map_border_and_empty_frame():
    """Sobel magnitude is normalised per frame; a constant frame gives 0 everywhere; 1-pixel-wide frames reflect to
    themselves."""
    rgb = torch.zeros(2, 3, 5, 1)
    rgb[1, :, 2] = 1.0
    e = alpha_oracle.sobel_edges_u8(rgb)
    assert e.shape == (2, 5, 1) and e[0].eq(0).all() and e[1].max() == 255


def _stub_engine(pipeline, preprocess, color_fix, shard, monkeypatch, calls):
    eng = object.__new__(pipeline.SeedVR2Engine)
    eng.device = torch.device("cpu")

    def fake_run(self, x, channels_last):                                  # (T,h,w,C) -> (3,T,Hp,Wp), nearest up-scale
        (H, W), _ = preprocess.resized_size(x.shape[1], x.shape[2], self.resolution, self.max_resolution)
        y = torch.nn.functional.interpolate(x[..., :3].permute(0, 3, 1, 2).float(), size=(H, W)).permute(1, 0, 2, 3)
        y = torch.nn.functional.pad(y, (0, (16 - W % 16) % 16, 0, (16 - H % 16) % 16))
        return (y * 2 - 1).to(torch.bfloat16)

    def fake_alpha(alpha, channel, sample, out=None):                      # alpha = the source frame's own marker
        assert alpha.shape[0] == sample.shape[0] and channel == alpha.shape[-1] - 1
        calls.append((alpha[:, 0, 0, channel].clone(), sample.shape))
        out.copy_(alpha[:, :1, :1, channel].expand(out.shape).to(out.dtype))
        return out

    monkeypatch.setattr(preprocess.VideoTransform, "run", fake_run)
    eng.vae_encode = lambda x: torch.zeros((x.shape[1] - 1) // 4 + 1, x.shape[2] // 8, x.shape[3] // 8, 16,
                                           dtype=torch.bfloat16)
    eng.inference = lambda noise, latent: noise
    eng.clip_workspace = lambda T, Hp, Wp: None
    eng.vae_decode = lambda z: torch.ones(3, 4 * z.shape[0] - 3, 8 * z.shape[1], 8 * z.shape[2], dtype=torch.bfloat16) * 0.5
    monkeypatch.setattr(color_fix, "sample_to_image",
                        lambda s_: (s_.float().permute(0, 2, 3, 1).clamp(-1, 1) * 0.5 + 0.5).to(torch.bfloat16))
    monkeypatch.setattr(shard, "blend_overlap", lambda p, c: ((p.float() + c.float()) / 2).to(p.dtype))
    alpha_mod = importlib.import_module("comfyui_seedvr2_videoupscaler_b200.alpha")
    monkeypatch.setattr(alpha_mod, "upscale_alpha", fake_alpha)
    return eng


def test_keep_alpha_control_flow_with_stubbed_kernels(pkg, monkeypatch):
    pipeline = importlib.import_module("comfyui_seedvr2_videoupscaler_b200.pipeline")
    preprocess = importlib.import_module("comfyui_seedvr2_videoupscaler_b200.preprocess")
    color_fix = importlib.import_module("comfyui_seedvr2_videoupscaler_b200.color_fix")
    shard = importlib.import_module("comfyui_seedvr2_videoupscaler_b200.shard")
    calls = []
    eng = _stub_engine(pipeline, preprocess, color_fix, shard, monkeypatch, calls)
    rgba = torch.rand(6, 20, 30, 4)
    rgba[..., 3] = (torch.arange(6).float() / 8).view(6, 1, 1)            # frame index as the alpha marker

    plain = eng.upscale_clip(rgba, resolution=40)                          # default: 4-channel input, 3-channel output
    assert plain.shape == (6, 40, 60, 3) and not calls
    out = eng.upscale_clip(rgba, resolution=40, keep_alpha=True)
    assert out.shape == (6, 40, 60, 4) and out.dtype == torch.bfloat16
    assert torch.equal(out[..., :3], plain)
    assert len(calls) == 1 and calls[0][1] == (6, 3, 40, 60)
    assert torch.equal(out[:, 0, 0, 3].float(), rgba[:, 0, 0, 3].bfloat16().float())
    rgb_only = eng.upscale_clip(rgba[..., :3], resolution=40, keep_alpha=True)
    assert rgb_only.shape == (6, 40, 60, 3) and len(calls) == 1

    # 13 frames, batch 5, overlap 2: batches [0,5) [3,8) [6,11) [9,13); written slices [0,5) [5,8) [8,11) [11,13)
    calls.clear()
    rgba = torch.rand(13, 20, 30, 4)
    rgba[..., 3] = (torch.arange(13).float() / 16).view(13, 1, 1)
    vid = eng.upscale_video(rgba, batch_size=5, temporal_overlap=2, resolution=40, keep_alpha=True)
    assert vid.shape == (13, 40, 60, 4)
    got = [(c[0] * 16).round().long().tolist() for c in calls]
    assert got == [[0, 1, 2, 3, 4], [5, 6, 7], [8, 9, 10], [11, 12]]
    assert torch.equal(vid[:, 0, 0, 3].float(), rgba[:, 0, 0, 3].bfloat16().float())
    plain_vid = eng.upscale_video(rgba, batch_size=5, temporal_overlap=2, resolution=40)
    assert plain_vid.shape == (13, 40, 60, 3) and torch.equal(vid[..., :3], plain_vid)


def test_alpha_host_mirror_refuses_cpu_tensors(pkg):
    alpha = importlib.import_module("comfyui_seedvr2_videoupscaler_b200.alpha")
    lib = importlib.import_module("comfyui_seedvr2_videoupscaler_b200.lib")
    with pytest.raises(lib.Svr2Error):
        alpha.edge_guided_alpha_upscale(torch.rand(1, 1, 4, 4), None, torch.rand(1, 3, 8, 8))
