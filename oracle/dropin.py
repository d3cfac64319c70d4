"""TEST INFRASTRUCTURE ONLY — the engine's model-slot modules as the reference's own pipeline objects see them.

``slot_engines`` builds ``B200NaDiT`` / ``B200VideoVAE`` on the CPU with the kernel layer replaced by the oracle (a test
double: there is no GPU where the reference pipeline runs).  Every slot call is bound against the real method's
signature before the double runs, so a keyword the engine does not accept fails the call, and is recorded.

``record_reference`` (run by ``python -m oracle.make_golden --dropin-only``, needs the reference tree) drives the
reference's ``VideoDiffusionInfer`` (``src/core/infer.py``) and memory manager (``src/optimization/memory_manager.py``)
with those modules in its slots and stores, in ``tests/golden/dropin_runner.npz``, the clip and its seeded inputs, every
slot call it made, what its phases returned and the module methods its lifecycle functions invoked.
``tests/test_dropin_reference_cpu.py`` checks the engine against that record without the reference.
"""
from __future__ import annotations

import importlib
import inspect
import json
import os
import sys
import types

import torch

DIT_OVERRIDES = dict(dim=256, heads=2, layers=4, mm_layers=2, txt_in_dim=64)
# nn.Module methods the reference's lifecycle functions may call on a model they are handed
MODULE_METHODS = ("named_modules", "modules", "children", "named_children", "parameters", "named_parameters", "buffers",
                  "named_buffers", "to", "cpu", "cuda", "half", "float", "zero_grad", "requires_grad_", "eval", "train",
                  "state_dict")


class Cfg(dict):
    """dict-backed stand-in for omegaconf.DictConfig: attribute access, .get, nested."""

    def __init__(self, d=None):
        super().__init__()
        for k, v in (d or {}).items():
            self[k] = Cfg(v) if isinstance(v, dict) else v

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:
            raise AttributeError(k) from e

    def __setattr__(self, k, v):
        self[k] = v


class ListCfg(list):
    pass


class Debug:
    def log(self, *a, **k):
        pass

    def start_timer(self, *a, **k):
        pass

    def end_timer(self, *a, **k):
        return 0.0

    def log_memory_state(self, *a, **k):
        pass


def _plain(v):
    """JSON form of a recorded call argument (tensors by shape and dtype, and their values when there are few)."""
    if isinstance(v, torch.Tensor):
        d = {"tensor": list(v.shape), "dtype": str(v.dtype).replace("torch.", "")}
        if v.numel() <= 8:
            d["values"] = v.flatten().tolist()
        return d
    if isinstance(v, (list, tuple)):
        return [_plain(x) for x in v]
    if isinstance(v, torch.device):
        return {"device": str(v)}
    if isinstance(v, torch.dtype):
        return {"dtype": str(v).replace("torch.", "")}
    return v


def unplain(v):
    """A recorded call argument back as a value (tensors stay descriptions: no recorded call passes one)."""
    if isinstance(v, list):
        return [unplain(x) for x in v]
    if isinstance(v, dict) and set(v) == {"device"}:
        return torch.device(v["device"])
    if isinstance(v, dict) and set(v) == {"dtype"}:
        return getattr(torch, v["dtype"])
    return v


def slot_engines(pkg, mp):
    """The slot modules with their forwards replaced by the oracle on the same weights; ``mp`` is a pytest MonkeyPatch."""
    from oracle import dit_oracle, vae_oracle
    lib = importlib.import_module("comfyui_seedvr2_videoupscaler_b200.lib")
    dit = importlib.import_module("comfyui_seedvr2_videoupscaler_b200.dit")
    vae = importlib.import_module("comfyui_seedvr2_videoupscaler_b200.vae")
    mp.setattr(lib, "device_check", lambda: (148, 10, 0))

    def fake_linear(a, w, *, bias=None, epi=0, **kw):          # the three load-time time-embedding GEMMs
        y = a.float() @ w.float().T + (bias.float() if bias is not None else 0)
        y = y.to(torch.bfloat16)
        return torch.nn.functional.silu(y.float()).to(torch.bfloat16) if epi & lib.EPI_SILU else y
    mp.setattr(lib, "linear", fake_linear)
    cfg = dit.dit_config("3b", **DIT_OVERRIDES)
    dsd = pkg.weights.synth_dit_state_dict(cfg, seed=1234, dtype=torch.float16)
    vsd = pkg.weights.synth_vae_state_dict(seed=4321, dtype=torch.float16)
    d, v = dit.B200NaDiT(cfg, dsd, device="cpu"), vae.B200VideoVAE(vsd, device="cpu")
    real = {"dit": dit.B200NaDiT.forward, "enc": vae.B200VideoVAE.encode, "dec": vae.B200VideoVAE.decode}
    calls = {"dit": [], "enc": [], "dec": []}
    contract = []
    ocfg = dit_oracle.dit_config("3b", **DIT_OVERRIDES)
    d32, v32 = {k: t.float() for k, t in dsd.items()}, {k: t.float() for k, t in vsd.items()}

    def bind(slot, self, args, kwargs):
        a = inspect.signature(real[slot]).bind(self, *args, **kwargs)
        a.apply_defaults()
        contract.append({"slot": slot, "positional": len(args), "keywords": sorted(kwargs),
                         "args": {k: _plain(x) for k, x in a.arguments.items() if k != "self"}})
        return a.arguments

    def dit_forward(self, *args, **kwargs):
        a = bind("dit", self, args, kwargs)
        vid, txt = a["vid"], a["txt"]
        vid_shape, txt_shape = torch.as_tensor(a["vid_shape"]).tolist(), torch.as_tensor(a["txt_shape"]).tolist()
        ts = a["timestep"]
        calls["dit"].append(dict(vid=tuple(vid.shape), txt=tuple(txt.shape), vid_shape=vid_shape, txt_shape=txt_shape,
                                 timestep=None if ts is None else torch.as_tensor(ts).tolist(), dtype=vid.dtype))
        (T, H, W), = vid_shape
        return dit.NaDiTOutput(dit_oracle.dit_forward(d32, ocfg, vid.float(), txt.float(), T, H, W).to(vid.dtype))

    def enc(self, *args, **kwargs):
        a = bind("enc", self, args, kwargs)
        x = a["x"]
        calls["enc"].append(dict(shape=tuple(x.shape), tiled=a["tiled"], tile_size=a["tile_size"],
                                 tile_overlap=a["tile_overlap"]))
        return vae.VAEOutput(latent=vae_oracle.vae_encode(v32, x.float()).to(x.dtype).squeeze(2), latent_dist=None)

    def dec(self, *args, **kwargs):
        a = bind("dec", self, args, kwargs)
        z = a["z"]
        calls["dec"].append(dict(shape=tuple(z.shape), tiled=a["tiled"], tile_size=a["tile_size"],
                                 tile_overlap=a["tile_overlap"]))
        z5 = z.unsqueeze(2) if z.ndim == 4 else z
        return vae.VAEOutput(sample=vae_oracle.vae_decode(v32, z5.float()).to(z.dtype).squeeze(2))
    mp.setattr(dit.B200NaDiT, "forward", dit_forward)
    mp.setattr(vae.B200VideoVAE, "encode", enc)
    mp.setattr(vae.B200VideoVAE, "decode", dec)
    return types.SimpleNamespace(dit=d, vae=v, calls=calls, contract=contract, real=real, d32=d32, v32=v32, ocfg=ocfg)


def trace_module_methods(mp, model, log):
    """Record every ``MODULE_METHODS`` call made on ``model`` (name, arguments) into ``log``; the calls still run."""
    for name in MODULE_METHODS:
        fn = getattr(model, name)

        def rec(*args, _fn=fn, _name=name, **kwargs):
            log.append({"method": _name, "args": _plain(list(args)), "kwargs": {k: _plain(v) for k, v in kwargs.items()}})
            return _fn(*args, **kwargs)
        mp.setattr(model, name, rec, raising=False)


# --------------------------------------------------------------------------------------------------------------------
# golden generation (needs the reference tree)
# --------------------------------------------------------------------------------------------------------------------
def _reference():
    import yaml
    from oracle import ref_import
    ref_import.install_stubs()
    om = types.ModuleType("omegaconf")
    om.DictConfig, om.ListConfig = Cfg, ListCfg
    om.OmegaConf = types.SimpleNamespace(load=lambda p: Cfg(yaml.safe_load(open(p))), create=lambda x: Cfg(x),
                                         register_new_resolver=lambda *a, **k: None)
    sys.modules.setdefault("omegaconf", om)
    infer = importlib.import_module("src.core.infer")
    mm = importlib.import_module("src.optimization.memory_manager")
    cfg = Cfg(yaml.safe_load(open(os.path.join(ref_import.REFERENCE_ROOT, "configs_3b", "main.yaml"))))
    cfg.vae.dtype = "bfloat16"
    cfg.diffusion.cfg.scale = 1.0                      # generation_phases.py:598-601: one-step, cfg 1
    cfg.diffusion.timesteps.sampling.steps = 1
    return infer, mm, cfg


# the runner as the test drives it: un-tiled encode, tiled decode with 64 x 64 tiles and 16-sample overlaps
RUNNER_KW = dict(encode_tiled=False, decode_tiled=True, decode_tile_size=(64, 64), decode_tile_overlap=(16, 16))


def record_reference(pkg, path):
    import numpy as np
    import pytest
    infer, mm, cfg = _reference()
    out = {}
    with pytest.MonkeyPatch.context() as mp:
        e = slot_engines(pkg, mp)
        runner = infer.VideoDiffusionInfer(cfg, Debug(), **RUNNER_KW)
        runner.dit, runner.vae = e.dit, e.vae
        runner.configure_diffusion(device=torch.device("cpu"), dtype=torch.bfloat16)
        g = torch.Generator().manual_seed(3)
        clip = (torch.rand(3, 5, 32, 48, generator=g) * 2 - 1).to(torch.bfloat16)         # c t h w (generation_phases.py:489)
        lat, = runner.vae_encode([clip])
        noise = torch.randn(lat.shape, generator=g).to(torch.bfloat16)
        cond = runner.get_condition(noise, task="sr", latent_blur=lat)
        txt = torch.randn(58, 64, generator=g).to(torch.bfloat16)
        x0, = runner.inference(noises=[noise], conditions=[cond], texts_pos=[txt], texts_neg=[txt])
        sample, = runner.vae_decode([x0])
        for k, t in dict(clip=clip, lat=lat, noise=noise, cond=cond, txt=txt, x0=x0, sample=sample).items():
            assert t.dtype == torch.bfloat16, k
            out[k] = t.float().numpy()                     # bf16 values are exact in float32
        contract = list(e.contract)
    lifecycle = {}
    with pytest.MonkeyPatch.context() as mp:
        e = slot_engines(pkg, mp)
        d, v = e.dit, e.vae
        for tag, fn in (("clear_rope_lru_caches", lambda: mm.clear_rope_lru_caches(d)),
                        ("manage_model_device", lambda: mm.manage_model_device(
                            model=d, target_device=torch.device("cpu"), model_name="DiT", debug=Debug(), reason="test"))):
            log = []
            with pytest.MonkeyPatch.context() as mq:
                trace_module_methods(mq, d, log)
                lifecycle[tag] = {"dit": log, "returned": fn()}
        runner = types.SimpleNamespace(dit=d, vae=v, sampler=1, schedule=1, sampling_timesteps=1)
        for tag, fn in (("cleanup_dit", lambda: mm.cleanup_dit(runner, debug=Debug(), cache_model=False)),
                        ("cleanup_vae", lambda: mm.cleanup_vae(runner, debug=Debug(), cache_model=False))):
            logs = {"dit": [], "vae": []}
            with pytest.MonkeyPatch.context() as mq:
                trace_module_methods(mq, d, logs["dit"])
                trace_module_methods(mq, v, logs["vae"])
                fn()
            lifecycle[tag] = logs
        assert runner.dit is None and runner.vae is None and runner.sampler is None
    meta = {"runner": {k: list(x) if isinstance(x, tuple) else x for k, x in RUNNER_KW.items()},
            "contract": contract, "lifecycle": lifecycle}
    np.savez_compressed(path, meta=np.array(json.dumps(meta, sort_keys=True)), **out)
    return meta
