"""CPU: the engine's model-slot modules against a record of the REFERENCE's own pipeline objects driving them.

``tests/golden/dropin_runner.npz`` was recorded (``python -m oracle.make_golden --dropin-only``, ``oracle/dropin.py``) by
running the reference's ``VideoDiffusionInfer`` (``src/core/infer.py``) with ``runner.dit`` / ``runner.vae`` set to the
engine's ``B200NaDiT`` / ``B200VideoVAE`` on one seeded clip, and its memory manager's lifecycle functions
(``src/optimization/memory_manager.py``) on those modules.  There is no GPU here, so the engine's kernel calls are replaced
by the (reference-pinned) oracle on the same weights.  What is under test is everything BETWEEN the reference and the
kernels: the call contract of the slots (``infer.py:117-199, 203-278, 315-395``: argument names, shapes, dtypes, the
``tiled`` / ``tile_size`` / ``tile_overlap`` keywords, ``.latent`` / ``.sample`` / ``.vid_sample``), the engine's own clip
runner (``pipeline.SeedVR2Engine``, which mirrors ``VideoDiffusionInfer``) against the reference runner's results, the
``nn.Module`` surface the pipeline relies on (``parameters()`` sniffing, ``named_modules()``, ``.to()``,
``requires_grad_().eval()``) and the lifecycle (``manage_model_device``, ``clear_rope_lru_caches``, ``cleanup_dit`` /
``release_model_memory``, ``memory_manager.py:427-455, 544-581, 670-738, 1011-1097``) as the module calls they make.
"""
import importlib
import inspect
import json
import os

import numpy as np
import pytest
import torch

from oracle import dropin

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "dropin_runner.npz")


@pytest.fixture(scope="module")
def gold():
    g = np.load(GOLD)
    t = {k: torch.from_numpy(g[k]).to(torch.bfloat16) for k in g.files if k != "meta"}     # bf16 values stored as f32
    return t, json.loads(str(g["meta"]))


@pytest.fixture()
def engines(pkg, monkeypatch):
    """B200NaDiT / B200VideoVAE built on the CPU with the kernel layer replaced by the oracle (test double)."""
    return dropin.slot_engines(pkg, monkeypatch)


def test_reference_runner_drives_the_engine_slots(pkg, engines, gold):
    """One clip through the reference's own VideoDiffusionInfer with the engine modules in its slots (as recorded), and
    the same clip through the engine's own runner."""
    from oracle import dit_oracle, vae_oracle
    t, meta = gold
    assert meta["runner"] == dict(encode_tiled=False, decode_tiled=True, decode_tile_size=[64, 64],
                                  decode_tile_overlap=[16, 16])
    # the calls the reference runner made, bound against the engine's real methods
    enc, dit_call, dec = meta["contract"]
    assert [c["slot"] for c in meta["contract"]] == ["enc", "dit", "dec"]
    modules = {"enc": engines.vae, "dit": engines.dit, "dec": engines.vae}
    for c in meta["contract"]:
        inspect.signature(engines.real[c["slot"]]).bind(modules[c["slot"]], *[None] * c["positional"],
                                                        **{k: None for k in c["keywords"]})
    assert enc["args"]["x"]["tensor"] == [1, 3, 5, 32, 48] and enc["args"]["tiled"] is False
    a = dit_call["args"]
    assert a["vid"]["tensor"] == [2 * 4 * 6, 33] and a["txt"]["tensor"] == [58, 64] and a["vid"]["dtype"] == "bfloat16"
    assert a["vid_shape"]["values"] == [2, 4, 6] and a["txt_shape"]["values"] == [58]
    assert a["timestep"]["values"] == [1000.0]                                              # the t the engine folds at load
    assert dec["args"]["z"]["tensor"] == [1, 16, 2, 4, 6]
    assert (dec["args"]["tiled"], dec["args"]["tile_size"], dec["args"]["tile_overlap"]) == (True, [64, 64], [16, 16])
    # what the reference runner returned, against the oracle
    assert tuple(t["lat"].shape) == (2, 4, 6, 16)                                           # t h w c, scaled by 0.9152
    assert (t["lat"].float() - vae_oracle.runner_encode(engines.v32, t["clip"][None].float())).abs().max() < 0.05
    vid = torch.cat([t["noise"], t["cond"]], -1).reshape(-1, 33).float()
    v = dit_oracle.dit_forward(engines.d32, engines.ocfg, vid, t["txt"].float(), 2, 4, 6)
    assert (t["x0"].float() - dit_oracle.one_step_latent(t["noise"].float(), v.view(2, 4, 6, 16))).abs().max() < 0.1
    assert tuple(t["sample"].shape) == (3, 5, 32, 48)
    # the engine's own runner on the same clip, noise and text reproduces the reference runner's phases: up to two bf16
    # ulps, since the oracle's fp32 sums on another CPU (other vector width, other thread count) round a few values the
    # other way
    pipeline = importlib.import_module("comfyui_seedvr2_videoupscaler_b200.pipeline")
    eng = object.__new__(pipeline.SeedVR2Engine)
    eng.device, eng.dit, eng.vae, eng.txt = torch.device("cpu"), engines.dit, engines.vae, t["txt"]
    for got, want in ((eng.vae_encode(t["clip"]), t["lat"]), (eng.inference(t["noise"], t["lat"]), t["x0"]),
                      (eng.vae_decode(t["x0"]), t["sample"])):
        assert got.dtype == torch.bfloat16
        torch.testing.assert_close(got.float(), want.float(), rtol=2 ** -6, atol=2 ** -8)
    assert [c["slot"] for c in engines.contract] == ["enc", "dit", "dec"]


def test_module_surface_and_lifecycle(engines, gold):
    _, meta = gold
    d, v = engines.dit, engines.vae
    for m in (d, v):
        assert isinstance(m, torch.nn.Module)
        p = next(m.parameters())                                  # device / dtype sniffing (generation_phases.py:620,708)
        assert p.device.type == "cpu" and p.dtype == torch.bfloat16 and not p.requires_grad
        assert len(list(m.buffers())) > 10
        m.requires_grad_(False).eval()                            # model_configuration.py:1240-1245
        assert m.to(torch.float16) is m and next(m.buffers()).dtype != torch.float16     # dtype casts are refused
        assert m.half() is m and m.float() is m
    # the attention seam is found the way apply_model_specific_config finds it (model_configuration.py:1206-1210)
    hits = [mod for mod in d.modules() if type(mod).__name__ == "FlashAttentionVarlen"]
    assert len(hits) == 1
    hits[0].attention_mode, hits[0].compute_dtype = "sdpa", torch.bfloat16
    # clear_rope_lru_caches counts the modules with a cached get_axial_freqs; it found none
    life = meta["lifecycle"]
    assert life["clear_rope_lru_caches"]["returned"] == 0
    assert not [n for n, mod in d.named_modules() if hasattr(getattr(mod, "get_axial_freqs", None), "cache_clear")]
    # manage_model_device moved nothing: the parameters already sit on the target device
    assert life["manage_model_device"]["returned"] is False and next(d.parameters()).device == torch.device("cpu")
    # every module call the lifecycle functions made, replayed on the engine modules: none fails, nothing is dropped
    n_buf = {id(m): sum(b.numel() for b in m.buffers()) for m in (d, v)}
    for tag in ("clear_rope_lru_caches", "manage_model_device", "cleanup_dit", "cleanup_vae"):
        for key, m in (("dit", d), ("vae", v)):
            for call in life[tag].get(key, []):
                r = getattr(m, call["method"])(*dropin.unplain(call["args"]),
                                               **{k: dropin.unplain(x) for k, x in call["kwargs"].items()})
                if inspect.isgenerator(r):
                    list(r)
    assert {c["method"] for c in life["cleanup_dit"]["dit"]} >= {"named_modules", "parameters", "zero_grad", "buffers"}
    for m in (d, v):
        assert sum(b.numel() for b in m.buffers()) == n_buf[id(m)]
    # offloaded / released weights must fail loudly, never fall back
    lib = importlib.import_module("comfyui_seedvr2_videoupscaler_b200.lib")
    with pytest.raises(lib.Svr2Error):
        d._require_cuda("forward")
