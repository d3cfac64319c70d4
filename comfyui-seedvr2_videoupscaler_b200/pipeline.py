"""Clip-level runner over the B200 engines.

Mirrors ``VideoDiffusionInfer`` (reference ``src/core/infer.py``): ``vae_encode``
(:117-199), ``inference`` (:315-395, one Euler step, cfg = 1: x0 = x_t - v,
``samplers/euler.py:59-63``), ``vae_decode`` (:203-278), with the latents handed
between phases on the device (no host bounce).  ``upscale_clip`` strings them
together the way ``generation_phases.py`` does for one clip: 4n+1 temporal pad
(:109-124), clamp + pad-16 + normalise (``generation_utils.py:72-84``), encode,
condition = [latent | 1] (``infer.py:54-78``), DiT, decode, crop, optional colour
correction against the input clip (``generation_phases.py:1249-1319``), [0,1] image format, and with ``keep_alpha`` the
edge-guided upscale of an RGBA clip's alpha (``generation_phases.py:1142-1217``).
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from . import alpha as alpha_ops
from . import color_fix, preprocess
from .dit import B200NaDiT, dit_config
from .vae import B200VideoVAE

SCALING_FACTOR = 0.9152   # configs_3b/main.yaml:60
SHIFTING_FACTOR = 0.0


def pad_4n1(n: int) -> int:
    """frames -> next 4n+1 (generation_phases.py:109-124)."""
    return n if n % 4 == 1 else n + (4 - (n - 1) % 4)


def pad_video_temporal(frames: torch.Tensor, count: int = 0, prepend: bool = False) -> torch.Tensor:
    """Temporal padding along dim 0 with REVERSED frames, the reference's single source of truth for the 4n+1
    constraint and for prepended frames (``pad_video_temporal``, generation_utils.py:598-657): ``count == 0`` pads the
    end up to the next 4n+1; the mirror excludes the edge frame itself ([f0..f7] -> [f0..f7, f6]); when more frames
    are needed than the clip has, the far-edge frame is repeated."""
    t = frames.shape[0]
    if count == 0 and not prepend:
        if t % 4 == 1:
            return frames
        count = ((t - 1) // 4 + 1) * 4 + 1 - t
    if count <= 0:
        return frames
    if count >= t:
        last = frames[-1:]
        repeated = last.expand(count - t + 1, *frames.shape[1:])
        rev = frames[1:].flip(0) if t > 1 else last[:0]
        return torch.cat([repeated, rev, frames] if prepend else [frames, rev, repeated], 0)
    rev = frames[1:count + 1].flip(0) if prepend else frames[-count - 1:-1].flip(0)
    return torch.cat([rev, frames] if prepend else [frames, rev], 0)


class SeedVR2Engine:
    def __init__(self, dit_cfg: dict, dit_sd: Dict[str, torch.Tensor], vae_sd: Dict[str, torch.Tensor],
                 txt_embed: torch.Tensor, device="cuda"):
        self.device = torch.device(device)
        self.dit = B200NaDiT(dit_cfg, dit_sd, device=device)
        self.vae = B200VideoVAE(vae_sd, device=device)
        self.txt = txt_embed.to(self.device, torch.bfloat16).contiguous()

    # ---- VideoDiffusionInfer.vae_encode ---------------------------------
    @torch.no_grad()
    def vae_encode(self, clip: torch.Tensor, workspace=None) -> torch.Tensor:
        """clip (3,T,H,W) in [-1,1] -> latent (T',h,w,16) bf16, scaled."""
        z = self.vae.encode(clip[None].to(self.device, torch.bfloat16), workspace=workspace).latent   # (1,16,T',h,w)
        z = (z - SHIFTING_FACTOR) * SCALING_FACTOR
        return z[0].permute(1, 2, 3, 0).contiguous()

    # ---- VideoDiffusionInfer.inference ------------------------------------
    @torch.no_grad()
    def inference(self, noise: torch.Tensor, latent: torch.Tensor, workspace=None) -> torch.Tensor:
        """noise, latent (T',h,w,16) -> x0 (T',h,w,16).  condition = cat[latent, 1] (task 'sr')."""
        T, h, w, c = latent.shape
        ones = torch.ones(T, h, w, 1, device=self.device, dtype=torch.bfloat16)
        vid = torch.cat([noise.to(self.device, torch.bfloat16), latent.to(torch.bfloat16), ones], -1)
        v = self.dit(vid.view(T * h * w, 2 * c + 1), self.txt, [[T, h, w]], [[self.txt.shape[0]]],
                     workspace=workspace).vid_sample
        return noise.to(self.device, torch.bfloat16) - v.view(T, h, w, c)

    # ---- VideoDiffusionInfer.vae_decode -----------------------------------
    @torch.no_grad()
    def vae_decode(self, latent: torch.Tensor, workspace=None) -> torch.Tensor:
        """latent (T',h,w,16) -> sample (3,T,H,W) bf16 in ~[-1,1]."""
        z = latent.permute(3, 0, 1, 2)[None]
        z = z / SCALING_FACTOR + SHIFTING_FACTOR
        return self.vae.decode(z, workspace=workspace).sample[0]

    def clip_workspace(self, T: int, Hp: int, Wp: int) -> Optional[torch.Tensor]:
        """ONE workspace for the three phases of a clip of T (4n+1) frames at Hp x Wp (multiples of 16): the maximum of
        the exact needs of VAE encode, the DiT forward and VAE decode (svr2_vae_workspace_bytes / svr2_workspace_bytes),
        with the VAE passes temporally sliced until they fit the free HBM.  The phases run one after the other on one
        stream, so they can share the bytes; the block is the engine's resident workspace (lib.workspace: kept between clips,
        grown on demand; the capture pool inside a CUDA graph).  None when a phase runs on the Python sequencing (profiling)."""
        from . import lib
        if not (self.vae._use_native() and self.dit.native and lib.PROFILER is None):
            return None
        Tl, h, w = (T - 1) // 4 + 1, Hp // 8, Wp // 8
        budget = int(0.92 * self.vae._free_bytes()) - 2 * 3 * T * Hp * Wp * 2      # the decoded clip and its crop
        need = max(self.vae.plan_slices(True, T, Hp, Wp, budget)[1], self.vae.plan_slices(False, Tl, h, w, budget)[1],
                   self.dit.workspace_bytes(Tl, h, w, self.txt.shape[0]))
        return lib.workspace(need, self.device)

    def latent_shape(self, frames: torch.Tensor, resolution: Optional[int] = None, max_resolution: int = 0):
        """(T', h, w, 16) of the latent ``upscale_clip`` will produce for ``frames`` (T,h,w,3)."""
        res = resolution if resolution is not None else min(frames.shape[1], frames.shape[2])
        H, W = preprocess.resized_size(frames.shape[1], frames.shape[2], res, max_resolution)[0]
        Hp, Wp = (H + 15) // 16 * 16, (W + 15) // 16 * 16
        return ((pad_4n1(frames.shape[0]) - 1) // 4 + 1, Hp // 8, Wp // 8, 16)

    def graphed(self, frames: torch.Tensor, **kw) -> "GraphedClip":
        """Capture ``upscale_clip`` for this clip shape into a CUDA graph (see ``GraphedClip``)."""
        return GraphedClip(self, frames, **kw)

    # ---- one clip end to end ------------------------------------------------
    @torch.no_grad()
    def upscale_clip(self, frames: torch.Tensor, noise: Optional[torch.Tensor] = None, seed: int = 42,
                     color_correction: str = "none", resolution: Optional[int] = None,
                     max_resolution: int = 0, keep_alpha: bool = False) -> torch.Tensor:
        """frames (T,h,w,C>=3) in [0,1]; ``resolution`` = target shortest edge (None: keep the size, i.e. the frames
        are already at the target resolution).  Returns (T,H,W,3) bf16 in [0,1] on the device.
        ``color_correction``: "none", "lab" (the reference CLI default), "wavelet" or "adain" — matched against the
        transformed input clip (generation_phases.py:1299-1317).
        ``keep_alpha`` with 4-channel frames: returns (T,H,W,4), the RGB of the 3-channel result plus channel 3 upscaled
        by ``alpha.upscale_alpha`` against the decoded sample before colour correction."""
        sample, style = self.clip_to_sample(frames, noise=noise, seed=seed, resolution=resolution,
                                            max_resolution=max_resolution)
        return self._finish(sample, style, color_correction, frames if keep_alpha else None)

    def _finish(self, sample: torch.Tensor, style: torch.Tensor, color_correction: str,
                frames: Optional[torch.Tensor]) -> torch.Tensor:
        """Phase 4 of one slice: with RGBA ``frames`` (the source frames of exactly this slice) the alpha is upscaled
        against the sample first, then colour correction and the [0,1] image format."""
        rgba = None
        if frames is not None and frames.shape[-1] == 4:
            src = frames if frames.is_cuda else frames[..., 3:].to(self.device)
            T, _, H, W = sample.shape
            rgba = torch.empty(T, H, W, 4, device=sample.device, dtype=torch.bfloat16)
            alpha_ops.upscale_alpha(src, src.shape[-1] - 1, sample, out=rgba[..., 3])
        if color_correction != "none":
            sample = color_fix.apply_color_correction(sample, style, color_correction)
        rgb = color_fix.sample_to_image(sample)                     # t h w c in [0,1]
        if rgba is None:
            return rgb
        rgba[..., :3] = rgb
        return rgba

    @torch.no_grad()
    def clip_to_sample(self, frames: torch.Tensor, noise: Optional[torch.Tensor] = None, seed: int = 42,
                       resolution: Optional[int] = None, max_resolution: int = 0):
        """Phases 1-3 for one clip: frames (T,h,w,3) in [0,1] -> (sample, style), both (T,3,H,W) bf16 in [-1,1]:
        the decoded clip and the transformed input clip it is colour-matched against in phase 4."""
        T0 = frames.shape[0]
        x = frames.to(self.device)
        x = pad_video_temporal(x)                                   # mirrored tail frames, generation_phases.py:109-124
        # resize (identity when the frames already have the target size) + clamp + pad-16 + normalise + c t h w
        # in one kernel (prepare_video_transforms, generation_utils.py:72-84)
        res = resolution if resolution is not None else min(frames.shape[1], frames.shape[2])
        tf = preprocess.VideoTransform(res, max_resolution)
        H0, W0 = tf.true_size(frames.shape[1], frames.shape[2])
        x = tf.run(x, channels_last=True)                           # (3, T, Hp, Wp) bf16 in [-1,1]
        ws = self.clip_workspace(x.shape[1], x.shape[2], x.shape[3])
        kw = {} if ws is None else {"workspace": ws}
        latent = self.vae_encode(x, **kw)
        if noise is None:
            g = torch.Generator(device=self.device).manual_seed(seed)
            noise = torch.randn(latent.shape, generator=g, device=self.device, dtype=torch.bfloat16)
        x0 = self.inference(noise, latent, **kw)
        y = self.vae_decode(x0, **kw)                               # (3,T,H,W)
        del ws, kw
        sample = y[:, :T0, :H0, :W0].permute(1, 0, 2, 3)            # t c h w, the layout of phase 4
        style = x[:, :T0, :H0, :W0].permute(1, 0, 2, 3)            # the transformed input clip in [-1,1]
        return sample, style

    @torch.no_grad()
    def upscale_video(self, frames: torch.Tensor, batch_size: int = 5, temporal_overlap: int = 0, seed: int = 42,
                      color_correction: str = "none", resolution: Optional[int] = None,
                      max_resolution: int = 0, keep_alpha: bool = False) -> torch.Tensor:
        """A whole video on one GPU the way the reference's four phases do it (generation_phases.py:271-289, 344-358,
        969-1000, 1236-1345): batches of ``batch_size`` frames stepping by ``batch_size - temporal_overlap``, every batch
        seeded identically, the overlap cross-faded into the previous batch's tail, colour correction per batch
        against its own input frames, [0,1] image format.  Returns (T,H,W,3) bf16, or (T,H,W,4) with ``keep_alpha``
        and 4-channel frames: each written slice's alpha comes from the source frames of that slice (the reference
        passes the whole batch's alpha and fails to broadcast when overlap frames were dropped or the batch was
        padded to 4n+1)."""
        from . import shard

        def clip(a, b):
            s, st = self.clip_to_sample(frames[a:b], seed=seed, resolution=resolution, max_resolution=max_resolution)
            return s.contiguous(), st.contiguous()

        written = [0]                           # run_batched post-processes the slices in order, laid end to end

        def post(sample, style):
            a = written[0]
            written[0] += sample.shape[0]
            return self._finish(sample, style, color_correction, frames[a:written[0]] if keep_alpha else None)

        return run_batched(frames.shape[0], batch_size, temporal_overlap, clip, shard.blend_overlap, post)



def batch_ranges(total: int, batch_size: int, temporal_overlap: int = 0):
    """([start, end) per batch, effective overlap) of generation_phases.py:271-289, 344-358: step =
    batch_size - overlap (overlap reset to 0 when it is not smaller than the batch); a trailing batch that would hold
    nothing but overlap frames is dropped."""
    step = batch_size - temporal_overlap if temporal_overlap > 0 else batch_size
    if step <= 0:
        step, temporal_overlap = batch_size, 0
    out = []
    for idx in range(0, total, step):
        end = min(idx + batch_size, total)
        if idx > 0 and end - idx <= temporal_overlap:
            break
        out.append((idx, end))
    return out, temporal_overlap


def run_batched(total: int, batch_size: int, temporal_overlap: int, clip_fn, blend_fn, post_fn) -> torch.Tensor:
    """The reference's batch loop with the engine plugged in as callables: ``clip_fn(start, end) -> (sample, style)``
    ((t,3,H,W) in [-1,1]), ``blend_fn(prev_tail, cur_head)``, ``post_fn(sample, style) -> (t,H,W,3)``.  Decoded batches are
    laid end to end; from the second batch on the first ``overlap`` frames are cross-faded into the tail already written
    and dropped (generation_phases.py:969-1000), and phase 4 then post-processes every batch's slice against its own
    input frames minus those overlap frames (:1249-1263)."""
    ranges, overlap = batch_ranges(total, batch_size, temporal_overlap)
    samples, styles = [], []
    written = 0
    for i, (a, b) in enumerate(ranges):
        sample, style = clip_fn(a, b)
        if i > 0 and overlap > 0 and overlap < sample.shape[0] and written >= overlap:
            # the tail lives in the previous batches' slices (it may span more than one when batches are short)
            tail = torch.cat(samples, 0)[-overlap:] if samples[-1].shape[0] < overlap else samples[-1][-overlap:]
            blended = blend_fn(tail.contiguous(), sample[:overlap].contiguous())
            k = overlap
            for j in range(len(samples) - 1, -1, -1):          # write the blended frames back, last slice first
                n = min(k, samples[j].shape[0])
                samples[j][samples[j].shape[0] - n:] = blended[k - n:k].to(samples[j].dtype)
                k -= n
                if k == 0:
                    break
            sample, style = sample[overlap:], style[overlap:]
        samples.append(sample)
        styles.append(style[: sample.shape[0]])
        written += sample.shape[0]
    return torch.cat([post_fn(s_, st_) for s_, st_ in zip(samples, styles)], 0)


class GraphedClip:
    """CUDA-graph replay of ``SeedVR2Engine.upscale_clip`` for one clip shape.

    The reference pays Python + launch overhead for every op of every clip (and so does the eager path here:
    ~3 000 kernel launches per 4K clip, ~1 700 for a single image, where the GPU work is shorter than the launch
    train).  All launches go through the C ABI on the current stream with pre-built tensor maps, nothing on the path
    synchronises with the host and the window / RoPE tables are cached per shape, so the whole clip — pre-processing,
    VAE encode, DiT, VAE decode, colour correction, formatting — captures into ONE graph whose intermediates live in
    the graph's private pool.  ``__call__`` copies the new frames into the static input and replays."""

    def __init__(self, engine: "SeedVR2Engine", frames: torch.Tensor, noise: Optional[torch.Tensor] = None,
                 seed: int = 42, warmup: int = 2, **clip_kwargs):
        from . import lib
        if lib.PROFILER is not None:
            raise lib.Svr2Error("per-call event profiling cannot run inside a graph capture")
        self.engine, self.kw = engine, clip_kwargs
        dev = engine.device
        self.static_in = frames.to(dev).clone()
        if noise is None:
            g = torch.Generator(device=dev).manual_seed(seed)
            noise = torch.randn(engine.latent_shape(frames, clip_kwargs.get("resolution"),
                                                    clip_kwargs.get("max_resolution", 0)),
                                generator=g, device=dev, dtype=torch.bfloat16)
        self.noise = noise.to(dev, torch.bfloat16).clone()
        if warmup > 0:                          # shape-dependent tables and kernel attributes (skip with warmup=0
            side = torch.cuda.Stream(device=dev)    # when the engine has already run this clip shape eagerly)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(warmup):
                    engine.upscale_clip(self.static_in, noise=self.noise, **clip_kwargs)
            torch.cuda.current_stream(dev).wait_stream(side)
        # the graph's private pool holds one whole clip of intermediates (~100 GB at 4K): hand the eager path's resident
        # workspace and cached blocks back first so both never have to coexist
        torch.cuda.synchronize(dev)
        lib.release_workspace(dev)
        torch.cuda.empty_cache()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.static_out = engine.upscale_clip(self.static_in, noise=self.noise, **clip_kwargs)

    def __call__(self, frames: torch.Tensor, clone: bool = False) -> torch.Tensor:
        """Replay on new frames of the captured shape.  The returned tensor is the graph's STATIC output buffer: the
        next replay overwrites it — pass ``clone=True`` (or copy it out, as bench.py does into pinned host memory)
        when results of several clips are kept."""
        if tuple(frames.shape) != tuple(self.static_in.shape):
            raise ValueError(f"GraphedClip captured frames of shape {tuple(self.static_in.shape)}, got {tuple(frames.shape)}")
        self.static_in.copy_(frames, non_blocking=True)
        self.graph.replay()
        return self.static_out.clone() if clone else self.static_out


def build_synthetic_engine(variant="3b", device="cuda", seed=1234, txt_len=58) -> SeedVR2Engine:
    """Random-init weights of the named architecture (no checkpoints exist offline)."""
    from . import weights
    cfg = dit_config(variant)
    dit_sd = weights.synth_dit_state_dict(cfg, seed=seed, dtype=torch.float16, device=device)
    vae_sd = weights.synth_vae_state_dict(seed=seed + 1, dtype=torch.float16, device=device)
    g = torch.Generator().manual_seed(seed + 2)
    txt = torch.randn(txt_len, cfg["txt_in_dim"], generator=g)
    eng = SeedVR2Engine(cfg, dit_sd, vae_sd, txt, device=device)
    del dit_sd, vae_sd
    return eng


def build_engine(dit_checkpoint: str, vae_checkpoint: str, txt_embed, device="cuda") -> SeedVR2Engine:
    """Engine from checkpoint files: DiT ``seedvr2_ema_{3b,7b}_{fp16,fp8_e4m3fn}.safetensors``, VAE
    ``ema_vae_fp16.safetensors`` (``model_registry.py:40-75``) and the positive text embedding (``pos_emb.pt``,
    ``generation_utils.py:load_text_embeddings``) given as a path or tensor."""
    from . import weights
    dit_sd = weights.load_state_dict(dit_checkpoint)
    cfg = dit_config(weights.detect_dit_variant(dit_sd))
    vae_sd = weights.load_state_dict(vae_checkpoint)
    txt = torch.load(txt_embed, map_location="cpu", weights_only=True) if isinstance(txt_embed, str) else txt_embed
    if txt.ndim == 3:
        txt = txt[0]
    return SeedVR2Engine(cfg, dit_sd, vae_sd, txt, device=device)
