"""RGBA alpha upscaling on the B200: csrc/alpha.cu against the reference's goldens and the torch oracle run on the same
GPU, CUDA-graph replays whose data flips the batch-wide decisions, the ``keep_alpha`` pipeline, and argument errors."""
import glob
import importlib
import os

import numpy as np
import pytest
import torch

from oracle import alpha_oracle

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ALPHA_GOLDENS = sorted(glob.glob(os.path.join(GOLD, "alpha_*.npz")))


@pytest.fixture(scope="module")
def mods(pkg):
    return (importlib.import_module("comfyui_seedvr2_videoupscaler_b200.alpha"),
            importlib.import_module("comfyui_seedvr2_videoupscaler_b200.lib"))


def stages(lib, alpha, rgb):
    """The three C-ABI stages on [T,1,h,w] alpha and [T,3,H,W] rgb -> (resized alpha, edges u8, final alpha fp32)."""
    T, _, h, w = alpha.shape
    H, W = rgb.shape[2:]
    dev = rgb.device
    need = lib.load().svr2_alpha_scratch_bytes(T, h, w, H, W)
    scratch = torch.empty(need, device=dev, dtype=torch.uint8)
    up = torch.empty(T, H, W, device=dev)
    edges = torch.empty(T, H, W, device=dev, dtype=torch.uint8)
    out = torch.empty(T, 1, H, W, device=dev)
    dt = {torch.float32: 0, torch.bfloat16: 1}[rgb.dtype]
    s = rgb.stride()
    lib.call("svr2_alpha_resize_f32", lib.ptr(alpha), {torch.float32: 0, torch.bfloat16: 1}[alpha.dtype], 0, 0, T, h, w, lib.ptr(up), H, W, lib.ptr(scratch), need,
             lib.stream())
    lib.call("svr2_alpha_edges_u8", lib.ptr(rgb), dt, s[1], s[0], s[2], T, h, w, H, W, lib.ptr(edges), lib.ptr(scratch),
             need, lib.stream())
    lib.call("svr2_alpha_refine", lib.ptr(rgb), dt, s[1], s[0], s[2], lib.ptr(up), lib.ptr(edges), T, h, w, H, W,
             lib.ptr(out), 0, 1, lib.ptr(scratch), need, lib.stream())
    return up, edges, out


def check_final(got, want, inter, binary, what):
    """<= 1e-5 everywhere for gradient alphas; for binary masks on >= 99.9 % of pixels, and every pixel beyond has an
    oracle q or pre-snap alpha within 1e-4 of a threshold (a 1-ulp difference there legitimately flips a snap)."""
    diff = (got.float() - want.float()).abs()
    bad = diff > 1e-5
    if not binary:
        assert not bad.any(), f"{what}: max |diff| {diff.max().item():.3g}"
        return
    assert bad.float().mean().item() <= 1e-3, f"{what}: {bad.sum().item()} pixels beyond 1e-5"
    near = torch.zeros_like(bad)
    for key in ("q", "mid"):
        v = inter[key].to(got.device)
        for th in (0.5, 0.3, 0.7):
            near |= (v - th).abs() <= 1e-4
    assert not (bad & ~near).any(), f"{what}: {(bad & ~near).sum().item()} pixels off without a threshold nearby"


def scene(T, h, w, H, W, binary=True, lo=-1.0, seed=0, dtype=torch.bfloat16):
    """Seeded RGBA scene on the GPU: a disc per frame (sharp for a binary mask, graded otherwise) whose RGB follows
    its outline, plus noise; rgb clamped to [lo, 1]."""
    g = torch.Generator(device="cuda").manual_seed(seed)

    def disc(hh, ww):
        yy, xx = torch.meshgrid(torch.linspace(-1, 1, hh, device="cuda"), torch.linspace(-1, 1, ww, device="cuda"),
                                indexing="ij")
        sh = torch.arange(T, device="cuda").view(T, 1, 1) * 0.05
        return ((xx - sh) ** 2 + (yy + sh) ** 2).sqrt()

    d = disc(h, w)
    alpha = (d < 0.6).float() if binary else (1.2 - d).clamp(0, 1)
    inside = (disc(H, W) < 0.6).float()[:, None]
    cin = torch.rand(T, 3, 1, 1, generator=g, device="cuda") * 2 - 1
    cout = torch.rand(T, 3, 1, 1, generator=g, device="cuda") * 2 - 1
    rgb = inside * cin + (1 - inside) * cout + 0.1 * torch.randn(T, 3, H, W, generator=g, device="cuda")
    return alpha[:, None].bfloat16(), rgb.clamp(lo, 1).to(dtype)


@pytest.mark.parametrize("path", ALPHA_GOLDENS, ids=lambda p: os.path.basename(p)[:-4])
def test_alpha_stages_match_golden(mods, path):
    _, lib = mods
    d = np.load(path)
    alpha, rgb = torch.from_numpy(d["alpha"]).cuda(), torch.from_numpy(d["rgb"]).cuda()
    up, edges, out = stages(lib, alpha, rgb)
    assert torch.equal(edges.cpu(), torch.from_numpy(d["edges_u8"]))
    ref, inter = alpha_oracle.edge_guided_alpha_upscale(alpha, rgb, intermediates=True)
    assert torch.equal(inter["edges_u8"], edges)
    assert (up - inter["alpha_up"][:, 0]).abs().max().item() <= 1e-6
    check_final(out, torch.from_numpy(d["out"]).cuda(), inter, bool(d["binary"]), "golden")
    check_final(out, ref, inter, bool(d["binary"]), "oracle")


def test_alpha_edges_bit_exact_at_4k(mods):
    _, lib = mods
    for lo in (-1.0, -1.5):                                   # one and two normalisations
        alpha, rgb = scene(2, 540, 960, 2160, 3840, lo=lo, seed=1)
        _, edges, _ = stages(lib, alpha, rgb)
        assert torch.equal(edges, alpha_oracle.sobel_edges_u8((rgb.float() + 1) / 2))


@pytest.mark.parametrize("binary", [True, False])
def test_alpha_4k_shard_vs_oracle(mods, binary):
    """The 4K shard: 8 x 720p alpha -> 2160 x 3840 against the decoded sample."""
    _, lib = mods
    alpha, rgb = scene(8, 720, 1280, 2160, 3840, binary=binary, seed=2)
    up, edges, out = stages(lib, alpha, rgb)
    ref, inter = alpha_oracle.edge_guided_alpha_upscale(alpha, rgb, intermediates=True)
    assert torch.equal(edges, inter["edges_u8"])
    assert (up - inter["alpha_up"][:, 0]).abs().max().item() <= 1e-6
    check_final(out, ref, inter, binary, "4k")


def test_alpha_graph_replay_follows_the_data(mods):
    """Captured on a binary mask with min(rgb) < 0; replayed on data that flips each decision it equals eager."""
    alpha_mod, _ = mods
    a0, r0 = scene(3, 48, 80, 96, 160, binary=True, lo=-1.0, seed=3)
    cases = {
        "gradient": scene(3, 48, 80, 96, 160, binary=False, lo=-1.0, seed=4),
        "rgb_nonneg": scene(3, 48, 80, 96, 160, binary=True, lo=0.0, seed=5),
        "rgb_below_m1": scene(3, 48, 80, 96, 160, binary=True, lo=-1.6, seed=6),
    }
    assert alpha_oracle.is_binary_mask(a0) and not alpha_oracle.is_binary_mask(cases["gradient"][0])
    assert cases["rgb_nonneg"][1].min() >= 0 and cases["rgb_below_m1"][1].min() < -1
    sa, sr = a0.clone(), r0.clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        alpha_mod.upscale_alpha(sa, None, sr)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        sout = alpha_mod.upscale_alpha(sa, None, sr)
    for name, (a, r) in [("capture", (a0, r0))] + list(cases.items()):
        sa.copy_(a)
        sr.copy_(r)
        graph.replay()
        eager = alpha_mod.upscale_alpha(a, None, r)
        assert torch.equal(sout, eager), name
        ref, inter = alpha_oracle.edge_guided_alpha_upscale(a, r, intermediates=True)
        check_final(eager, ref, inter, alpha_oracle.is_binary_mask(a), name)


def test_alpha_entry_points_layouts(mods):
    """[T,h,w,4] frames with the alpha at channel 3 and a [T,H,W,4] bf16 destination equal the [T,1,h,w] path."""
    alpha_mod, _ = mods
    a, r = scene(2, 30, 44, 55, 80, seed=7)
    frames = torch.rand(2, 30, 44, 4, device="cuda")
    frames[..., 3] = a[:, 0].float()
    want = alpha_mod.edge_guided_alpha_upscale(a, None, r)
    rgba = torch.zeros(2, 55, 80, 4, device="cuda", dtype=torch.bfloat16)
    alpha_mod.upscale_alpha(frames, 3, r, out=rgba[..., 3])
    assert torch.equal(rgba[..., 3], want[:, 0].bfloat16()) and rgba[..., :3].eq(0).all()
    planes = r.permute(1, 0, 2, 3).contiguous().permute(1, 0, 2, 3)       # strided [T,3,H,W] view of [3,T,H,W]
    assert torch.equal(alpha_mod.upscale_alpha(a, None, planes), want)
    rgba_list = alpha_mod.process_alpha_for_batch([r], a, None, "cuda", torch.bfloat16)
    assert rgba_list[0].shape == (2, 4, 55, 80) and torch.equal(rgba_list[0][:, 3:], want.bfloat16())


def test_alpha_errors_return_status(mods):
    alpha_mod, lib = mods
    L = lib.load()
    a, r = scene(2, 16, 16, 32, 32, seed=8)
    up = torch.empty(2, 32, 32, device="cuda")
    small = torch.empty(64, device="cuda", dtype=torch.uint8)
    rc = L.svr2_alpha_resize_f32(lib.ptr(a), 1, 0, 0, 2, 16, 16, lib.ptr(up), 32, 32, lib.ptr(small), 64, lib.stream())
    assert rc != 0 and b"scratch" in L.svr2_last_error()
    need = L.svr2_alpha_scratch_bytes(2, 16, 16, 32, 32)
    scratch = torch.empty(need, device="cuda", dtype=torch.uint8)
    rc = L.svr2_alpha_resize_f32(lib.ptr(a), 1, 4, 4, 2, 16, 16, lib.ptr(up), 32, 32, lib.ptr(scratch), need, lib.stream())
    assert rc != 0 and b"channel" in L.svr2_last_error()
    edges = torch.empty(2, 32, 32, device="cuda", dtype=torch.uint8)
    s = r.stride()
    rc = L.svr2_alpha_edges_u8(lib.ptr(r), 7, s[1], s[0], s[2], 2, 16, 16, 32, 32, lib.ptr(edges), lib.ptr(scratch), need,
                               lib.stream())
    assert rc != 0
    rc = L.svr2_alpha_refine(lib.ptr(r), 1, s[1], s[0], 8, lib.ptr(up), lib.ptr(edges), 2, 16, 16, 32, 32, lib.ptr(up), 0,
                             1, lib.ptr(scratch), need, lib.stream())
    assert rc != 0 and b"stride" in L.svr2_last_error()
    with pytest.raises(ValueError):
        alpha_mod.edge_guided_alpha_upscale(a, None, r[:1])
    with pytest.raises(lib.Svr2Error):                        # a 40x down-scale needs more taps than the tables hold
        alpha_mod.edge_guided_alpha_upscale(torch.rand(2, 1, 320, 320, device="cuda"), None, r[:, :, :8, :8])
    torch.cuda.synchronize()


def _engine(pkg):
    pipeline = importlib.import_module("comfyui_seedvr2_videoupscaler_b200.pipeline")
    dit = importlib.import_module("comfyui_seedvr2_videoupscaler_b200.dit")
    cfg = dit.dit_config("3b", dim=256, heads=2, layers=2, mm_layers=1, txt_in_dim=64)
    return pipeline.SeedVR2Engine(cfg, pkg.weights.synth_dit_state_dict(cfg, seed=1),
                                  pkg.weights.synth_vae_state_dict(seed=2), torch.randn(58, 64))


def test_pipeline_keep_alpha_clip_and_graph(pkg, mods):
    alpha_mod, _ = mods
    eng = _engine(pkg)
    g = torch.Generator().manual_seed(0)
    rgba = torch.rand(5, 36, 52, 4, generator=g).cuda()
    rgba[..., 3] = (rgba[..., 3] > 0.5).float()
    rgba2 = torch.rand(5, 36, 52, 4, generator=g).cuda()
    kw = dict(resolution=72, color_correction="lab")
    noise = torch.randn(eng.latent_shape(rgba, 72), generator=torch.Generator().manual_seed(1)).cuda()
    plain = eng.upscale_clip(rgba, noise=noise, **kw).clone()
    out = eng.upscale_clip(rgba, noise=noise, keep_alpha=True, **kw).clone()
    assert plain.shape == (5, 72, 104, 3) and out.shape == (5, 72, 104, 4) and out.dtype == torch.bfloat16
    assert torch.equal(out[..., :3], plain)
    sample, _ = eng.clip_to_sample(rgba, noise=noise, resolution=72)
    want = alpha_mod.edge_guided_alpha_upscale(rgba[..., 3][:, None], None, sample)
    assert torch.equal(out[..., 3], want[:, 0].bfloat16())
    assert torch.equal(eng.upscale_clip(rgba[..., :3], noise=noise, keep_alpha=True, **kw), plain)
    eager2 = eng.upscale_clip(rgba2, noise=noise, keep_alpha=True, **kw).clone()
    gc = eng.graphed(rgba, noise=noise, keep_alpha=True, **kw)
    assert torch.equal(gc(rgba), out)
    assert torch.equal(gc(rgba2), eager2)                     # the second clip's alpha is a gradient: r = 3 on replay


def test_pipeline_keep_alpha_video(pkg):
    eng = _engine(pkg)
    rgba = torch.rand(13, 36, 52, 4, generator=torch.Generator().manual_seed(2)).cuda()
    kw = dict(resolution=72, color_correction="wavelet")
    vid = eng.upscale_video(rgba, batch_size=5, temporal_overlap=2, keep_alpha=True, **kw)
    assert vid.shape == (13, 72, 104, 4) and torch.isfinite(vid.float()).all()
    assert 0 <= vid.min() and vid.max() <= 1
    assert torch.equal(vid[..., :3], eng.upscale_video(rgba, batch_size=5, temporal_overlap=2, **kw))
    plain = eng.upscale_video(rgba, batch_size=5, temporal_overlap=0, keep_alpha=True, **kw)
    assert plain.shape == (13, 72, 104, 4)
    assert torch.equal(plain[:5], eng.upscale_clip(rgba[:5], keep_alpha=True, **kw))
