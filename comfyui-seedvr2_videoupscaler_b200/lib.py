"""ctypes binding of csrc/libsvr2.so (include/svr2.h).

PyTorch tensors supply device memory (`data_ptr()`) and the current stream only.
There is deliberately no fallback: if the library is missing or a call fails, we raise.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_float, c_int, c_int64, c_void_p, POINTER

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SVR2_LIB") or os.path.join(HERE, "csrc", "libsvr2.so")   # SVR2_LIB: another build (A/B tools only)

EPI_BIAS, EPI_GATE, EPI_RESIDUAL, EPI_SWIGLU, EPI_GELU, EPI_F32, EPI_SILU = 1, 2, 4, 8, 16, 32, 128
EPI_ROWSTAT, EPI_PEXP, EPI_ROWSCALE = 256, 512, 1024

class ModelDesc(ctypes.Structure):
    """svr2_model_desc (include/svr2.h)"""
    _fields_ = [("variant", c_int), ("dim", c_int), ("heads", c_int), ("layers", c_int), ("mm_layers", c_int),
                ("txt_in_dim", c_int), ("in_ch", c_int), ("out_ch", c_int), ("mlp_kind", c_int), ("mlp_hidden", c_int),
                ("out_norm", c_int), ("last_vid_only", c_int), ("eps", c_float), ("timestep", c_float)]


class TensorDesc(ctypes.Structure):
    """svr2_tensor_desc (include/svr2.h)"""
    _fields_ = [("name", ctypes.c_char_p), ("data", c_void_p), ("dtype", c_int), ("rank", c_int), ("shape", c_int64 * 5)]


# name -> argtypes; every function returns int (svr2_status) except svr2_last_error
_P = c_void_p
SIGNATURES = {
    "svr2_version": [],
    "svr2_set_cta_pair": [c_int],
    "svr2_set_conv_wreuse": [c_int],
    "svr2_device_check": [POINTER(c_int), POINTER(c_int), POINTER(c_int)],
    "svr2_create": [POINTER(c_void_p), c_int, POINTER(ModelDesc)],
    "svr2_destroy": [_P],
    "svr2_load_weights": [_P, POINTER(TensorDesc), ctypes.c_size_t, c_int],
    "svr2_workspace_bytes": [_P, c_int, c_int, c_int, c_int],
    "svr2_dit_forward": [_P, _P, _P, c_int, c_int, c_int, c_int, _P, _P],
    "svr2_dit_forward_ws": [_P, _P, _P, c_int, c_int, c_int, c_int, _P, _P, ctypes.c_size_t, _P],
    "svr2_vae_workspace_bytes": [_P, c_int, c_int, c_int, c_int, c_int],
    "svr2_vae_encode": [_P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, ctypes.c_size_t, _P],
    "svr2_vae_decode": [_P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, ctypes.c_size_t, _P],
    "svr2_vae_last_launches": [_P],
    "svr2_linear_bf16": [_P, c_int64, _P, c_int64, c_int, c_int, c_int, c_int, _P, _P, _P, _P, c_int64, c_float, _P],
    "svr2_conv3d_bf16": [_P, c_int, c_int, c_int, c_int, _P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                         c_int, _P, _P, _P, c_int, c_int, c_int, _P],
    "svr2_conv3d_stats_bf16": [_P, c_int, c_int, c_int, c_int, _P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                               c_int, _P, _P, _P, c_int, c_int, c_int, _P, c_int64, POINTER(c_int), _P],
    "svr2_conv3d_shortcut_stats_bf16": [_P, c_int, c_int, c_int, c_int, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, c_int,
                                        _P, c_int, c_int, _P, c_int64, POINTER(c_int), _P],
    "svr2_conv_stat_slots": [c_int, c_int, c_int],
    "svr2_groupnorm_from_stats_bf16": [_P, _P, c_int, c_int, c_int, _P, _P, c_float, c_int, c_int, c_int, _P, c_int, _P,
                                       _P],
    "svr2_upsample_shuffle_bf16": [_P, c_int, c_int, c_int, c_int, _P, _P, c_int, c_int, _P, c_int, c_int, _P],
    "svr2_attn_varlen_bf16": [_P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, _P, _P],
    "svr2_rmsnorm_ada_bf16": [_P, _P, c_int, c_int, c_float, _P, _P, _P, c_int, _P],
    "svr2_qk_norm_rope_window_bf16": [_P, _P, _P, _P, _P, _P, c_int, _P, _P, _P, _P, c_float, c_int, c_int, _P, _P,
                                      _P, _P],
    "svr2_qk_norm_rope_rows_bf16": [_P, _P, _P, _P, _P, _P, c_int, _P, _P, _P, _P, c_float, _P, c_int, c_int, _P, _P,
                                    _P, _P],
    "svr2_linear_qkv_rope_bf16": [_P, c_int64, _P, c_int64, c_int, c_int, c_int, _P, _P, _P, _P, c_int, _P, c_float, _P,
                                  _P, _P, _P],
    "svr2_txt_window_mean_bf16": [_P, _P, c_int, c_int, c_int, _P],
    "svr2_patchify_bf16": [_P, _P, c_int, c_int, c_int, c_int, c_int, _P],
    "svr2_unpatchify_bf16": [_P, c_int, _P, c_int, c_int, c_int, c_int, _P],
    "svr2_groupnorm_bf16": [_P, _P, c_int, c_int, c_int, _P, _P, c_float, c_int, c_int, c_int, _P, c_int64, _P],
    "svr2_groupnorm_scratch_bytes": [c_int, c_int, c_int],
    "svr2_softmax_rows_bf16": [_P, c_int64, _P, c_int64, c_int, c_int, _P],
    "svr2_linear_ex_bf16": [_P, c_int64, _P, c_int64, c_int, c_int, c_int, c_int, _P, _P, _P, _P, c_int64, c_float, _P, _P,
                            c_int64, _P, _P],
    "svr2_rowstat_max": [_P, c_int, c_int64, _P, c_int, _P, _P],
    "svr2_pexp_stat_combine": [_P, c_int, c_int64, _P, _P, c_int, _P, _P],
    "svr2_rowstat_slots": [c_int],
    "svr2_rowstat_combine": [_P, c_int, c_int64, _P, c_int, _P],
    "svr2_transpose_bf16": [_P, c_int64, _P, c_int64, c_int, c_int, _P],
    "svr2_ncdhw_to_ndhwc_bf16": [_P, c_int, c_int, c_int, c_int, c_int, _P, c_int, c_int, c_float, _P],
    "svr2_ndhwc_to_ncdhw": [_P, c_int, c_int, c_int, c_int, c_int, _P, c_int, _P],
    "svr2_conv_tap_gather": [_P, c_int64, c_int, _P, c_int, c_int, c_int, _P, c_int, _P],
    "svr2_im2col3_bf16": [_P, c_int, c_int, c_int, c_int, c_int, _P, c_int, _P],
    "svr2_wavelet_level_bf16": [_P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P],
    "svr2_adain_bf16": [_P, _P, _P, c_int, c_int64, _P, _P],
    "svr2_rgb_to_lab_f32": [_P, _P, c_int, c_int64, _P],
    "svr2_lab_to_rgb_bf16": [_P, _P, _P, _P, c_float, _P, c_int, c_int64, _P],
    "svr2_histogram_match_scratch_bytes": [c_int64],
    "svr2_histogram_match_f32": [_P, _P, _P, c_int64, _P, c_int64, _P],
    "svr2_sample_to_image_bf16": [_P, _P, c_int, c_int64, _P],
    "svr2_blend_overlap_bf16": [_P, _P, _P, _P, _P, c_int, c_int64, _P],
    "svr2_blend_overlap_f32": [_P, _P, _P, _P, _P, c_int, c_int64, _P],
    "svr2_tile_accumulate_bf16": [_P, c_int64, c_int, c_int, c_int, c_int, _P, _P, _P, _P, c_int, c_int, c_int, c_int, _P],
    "svr2_tile_normalize_bf16": [_P, _P, c_int, c_int64, _P],
    "svr2_resize_scratch_bytes": [c_int, c_int, c_int, c_int],
    "svr2_resize_bicubic_aa_bf16": [_P, c_int, c_int, c_int, c_int, c_int, c_int, _P, c_int, c_int, c_int, _P, c_int64,
                                    _P],
    "svr2_alpha_scratch_bytes": [c_int, c_int, c_int, c_int, c_int],
    "svr2_alpha_resize_f32": [_P, c_int, c_int, c_int, c_int, c_int, c_int, _P, c_int, c_int, _P, c_int64, _P],
    "svr2_alpha_edges_u8": [_P, c_int, c_int64, c_int64, c_int64, c_int, c_int, c_int, c_int, c_int, _P, _P, c_int64, _P],
    "svr2_alpha_refine": [_P, c_int, c_int64, c_int64, c_int64, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, c_int,
                          c_int, _P, c_int64, _P],
}

_lib = None


class Svr2Error(RuntimeError):
    pass


def load() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise Svr2Error(f"{LIB_PATH} not built — run `python __graft_entry__.py` (build()); "
                            "there is no CPU / PyTorch fallback")
        lib = ctypes.CDLL(LIB_PATH)
        lib.svr2_last_error.restype = ctypes.c_char_p
        lib.svr2_last_error.argtypes = []
        lib.svr2_engine_last_error.restype = ctypes.c_char_p
        lib.svr2_engine_last_error.argtypes = [c_void_p]
        for name, args in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = c_int64 if (name.endswith("_bytes") or name == "svr2_vae_last_launches") else (None if name in ("svr2_set_cta_pair", "svr2_set_conv_wreuse", "svr2_destroy") else c_int)
            fn.argtypes = args
        _lib = lib
    return _lib


def _check(rc: int, what: str):
    if rc != 0:
        raise Svr2Error(f"{what} failed ({rc}): {load().svr2_last_error().decode()}")


def ptr(t):
    return None if t is None else c_void_p(t.data_ptr())


def stream():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


# kernels launched per C-ABI call (for the bench's gpu_launches count)
KERNELS_PER_CALL = {"svr2_groupnorm_bf16": 3, "svr2_groupnorm_from_stats_bf16": 2,
                    "svr2_resize_bicubic_aa_bf16": 3,      # two tap-table kernels + the resize
                    "svr2_adain_bf16": 2,                  # statistics + apply
                    "svr2_histogram_match_f32": 2,         # iota + rank scatter (the CUB radix-sort passes are library launches)
                    "svr2_alpha_resize_f32": 4,            # two tap-table kernels + the binary-mask count + the resize
                    "svr2_alpha_edges_u8": 2,              # flags / per-frame maxima + the edge map
                    "svr2_alpha_refine": 2}                # the two guided-filter box passes


class Profiler:
    """Optional per-call CUDA-event timing on the launching stream (bench.py roofline).
    Off by default: `lib.PROFILER = Profiler()` turns it on."""

    def __init__(self):
        self.records = []      # (name, flops, bytes, start_event, end_event)
        self.launches = 0
        self.detail = False    # tag GEMM/conv records with their shapes

    def summary(self):
        torch.cuda.synchronize()
        out = {}
        for name, flops, nbytes, e0, e1 in self.records:
            d = out.setdefault(name, dict(calls=0, ms=0.0, flops=0.0, bytes=0.0))
            d["calls"] += 1
            d["ms"] += e0.elapsed_time(e1)
            d["flops"] += flops
            d["bytes"] += nbytes
        return out

    def reset(self):
        self.records.clear()
        self.launches = 0


PROFILER = None
LAUNCHES = 0


def call(name: str, *args, flops: float = 0.0, nbytes: float = 0.0, tag: str = ""):
    global LAUNCHES
    LAUNCHES += KERNELS_PER_CALL.get(name, 1)
    prof = PROFILER
    if prof is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _check(getattr(load(), name)(*args), name)
        e1.record()
        prof.records.append((name + tag, flops, nbytes, e0, e1))
    else:
        _check(getattr(load(), name)(*args), name)


def device_check():
    sm, maj, mnr = c_int(), c_int(), c_int()
    _check(load().svr2_device_check(ctypes.byref(sm), ctypes.byref(maj), ctypes.byref(mnr)), "svr2_device_check")
    return sm.value, maj.value, mnr.value


# --------------------------------------------------------------------------
# thin tensor-level wrappers (shape checks + output allocation only)
# --------------------------------------------------------------------------
def _bf16c(t, name):
    assert t.dtype == torch.bfloat16 and t.is_cuda, f"{name}: bf16 CUDA tensor required"
    return t


def linear(a, w, *, bias=None, gate=None, residual=None, epi=0, out=None, out_scale=1.0, n_valid=None,
           count_flops=True, rowscale=None, stat_out=None, run_if=None):
    """out = epi(a @ w^T).  a [M,K] (row stride lda), w [N,K]."""
    _bf16c(a, "a"), _bf16c(w, "w")
    M, K = a.shape
    N = w.shape[0]
    assert a.stride(1) == 1 and w.stride(1) == 1
    if bias is not None:
        epi |= EPI_BIAS
    if gate is not None:
        if not epi & EPI_PEXP:
            epi |= EPI_GATE
        assert gate.dtype == torch.float32
    if residual is not None:
        epi |= EPI_RESIDUAL
    n_out = N // 2 if epi & EPI_SWIGLU else N
    if out is None:
        out = torch.empty(M, n_out, device=a.device, dtype=torch.float32 if epi & EPI_F32 else torch.bfloat16)
    if residual is not None:
        assert residual.stride(0) == out.stride(0)
    ldc = out.stride(0) // 2 if epi & EPI_ROWSTAT else out.stride(0)   # ROWSTAT: float2 slots per row
    extras = ()
    name = "svr2_linear_bf16"
    if rowscale is not None or stat_out is not None or run_if is not None:
        name = "svr2_linear_ex_bf16"
        if rowscale is not None:
            epi |= EPI_ROWSCALE
        extras = (ptr(rowscale), ptr(stat_out), stat_out.stride(0) // 2 if stat_out is not None else 0, ptr(run_if))
    call(name, ptr(a), a.stride(0), ptr(w), w.stride(0), M, N, K, epi, ptr(bias), ptr(gate),
         ptr(residual), ptr(out), ldc, float(out_scale), *extras, stream(),
         flops=2.0 * M * (n_valid if n_valid is not None else N) * K if count_flops else 0.0,
         tag=f"|{M}x{N}x{K}|e{epi}" if (PROFILER is not None and PROFILER.detail) else "")
    return out


def attn_varlen(q, k, v, cu_seqlens, max_seqlen, out=None, out_row_map=None, flops=0.0):
    _bf16c(q, "q"), _bf16c(k, "k"), _bf16c(v, "v")
    total, heads, d = q.shape
    assert d == 128 and q.is_contiguous() and k.is_contiguous() and v.is_contiguous()
    assert cu_seqlens.dtype == torch.int32 and cu_seqlens.is_cuda
    if out is None:
        out = torch.empty_like(q)
    call("svr2_attn_varlen_bf16", ptr(q), ptr(k), ptr(v), ptr(out), ptr(cu_seqlens), cu_seqlens.numel() - 1, total,
         heads, int(max_seqlen), ptr(out_row_map), stream(), flops=float(flops))
    return out


def rmsnorm_ada(x, scale, shift, *, weight=None, mode=0, eps=1e-5, out=None):
    _bf16c(x, "x")
    rows, dim = x.shape
    assert x.is_contiguous()
    if out is None:
        out = torch.empty_like(x)
    call("svr2_rmsnorm_ada_bf16", ptr(x), ptr(out), rows, dim, float(eps), ptr(weight), ptr(scale), ptr(shift),
         int(mode), stream(), nbytes=4.0 * rows * dim)
    return out


def conv3d(x, T_in_total, H, W, Cin, w, Cout, k, stride_t, stride_hw, pad_hw, T_out, y, *, bias=None, residual=None,
           out_t_pad=0, out_dup_head=0, ldc=None):
    epi = (EPI_BIAS if bias is not None else 0) | (EPI_RESIDUAL if residual is not None else 0)
    call("svr2_conv3d_bf16", ptr(x), T_in_total, H, W, Cin, ptr(w), Cout, k[0], k[1], k[2], stride_t, stride_hw,
         pad_hw, T_out, epi, ptr(bias), ptr(residual), ptr(y), out_t_pad, out_dup_head,
         int(ldc if ldc is not None else Cout), stream(),
         flops=2.0 * T_out * (H // stride_hw) * (W // stride_hw) * Cout * k[0] * k[1] * k[2] * Cin)
    return y


# --------------------------------------------------------------------------
# engine workspace: ONE resident block per device for the native runtimes (a clip's encode / DiT / decode phases share it)
# --------------------------------------------------------------------------
_WORKSPACES = {}


def workspace(nbytes: int, device) -> torch.Tensor:
    """uint8 CUDA tensor of >= nbytes.  Outside a CUDA-graph capture the block is kept resident and reused (grown when
    a larger clip arrives): handing ~100 GB back to the caching allocator after every clip lets other allocations land
    inside the freed segment, and the next clip's request then neither fits the fragments nor a fresh cudaMalloc.
    Inside a capture the block comes from the graph's private pool.  One stream at a time uses the block."""
    device = torch.device(device)
    if torch.cuda.is_current_stream_capturing():
        return torch.empty(nbytes, device=device, dtype=torch.uint8)
    key = device.index if device.index is not None else torch.cuda.current_device()
    t = _WORKSPACES.get(key)
    if t is None or t.numel() < nbytes:
        if t is not None:
            del t
            release_workspace(device)
        try:
            t = torch.empty(nbytes, device=device, dtype=torch.uint8)
        except torch.OutOfMemoryError:
            torch.cuda.synchronize(device)
            torch.cuda.empty_cache()
            t = torch.empty(nbytes, device=device, dtype=torch.uint8)
        _WORKSPACES[key] = t
    return t


def workspace_held(device) -> int:
    device = torch.device(device)
    t = _WORKSPACES.get(device.index if device.index is not None else torch.cuda.current_device())
    return 0 if t is None else t.numel()


def release_workspace(device=None) -> None:
    """Drop the resident block(s) — before a CUDA-graph capture of a clip (its pool holds its own) or when another
    consumer needs the HBM."""
    if device is None:
        keys = list(_WORKSPACES)
        _WORKSPACES.clear()
    else:
        device = torch.device(device)
        key = device.index if device.index is not None else torch.cuda.current_device()
        keys = [key] if _WORKSPACES.pop(key, None) is not None else []
    had = bool(keys)
    # back to the DRIVER, not to the caching allocator: a cached ~100 GB segment gets split by whatever is allocated next,
    # and one small long-lived tensor inside it keeps the whole segment from ever being handed out again in one piece
    if had and not torch.cuda.is_current_stream_capturing():
        for k in keys:
            torch.cuda.synchronize(k)
        torch.cuda.empty_cache()


# --------------------------------------------------------------------------
# handle API (native host runtime, csrc/engine.cu)
# --------------------------------------------------------------------------
_TORCH_DT = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}


def engine_create(desc: ModelDesc, device_index: int) -> c_void_p:
    h = c_void_p()
    _check(load().svr2_create(ctypes.byref(h), int(device_index), ctypes.byref(desc)), "svr2_create")
    return h


def engine_load(handle: c_void_p, tensors: dict, copy: bool) -> None:
    """tensors: engine-layout name -> torch tensor (CUDA tensors are borrowed when copy is False; host tensors need copy)."""
    items = [(k, t.contiguous()) for k, t in tensors.items()]
    arr = (TensorDesc * len(items))()
    for d, (k, t) in zip(arr, items):
        d.name, d.data, d.dtype, d.rank = k.encode(), t.data_ptr(), _TORCH_DT[t.dtype], max(t.ndim, 1)
        for i, n in enumerate(t.shape if t.ndim else (1,)):
            d.shape[i] = n
    _check(load().svr2_load_weights(handle, arr, len(items), int(copy)), "svr2_load_weights")
    if copy:
        torch.cuda.synchronize()          # the sources may be temporaries


def engine_destroy(handle) -> None:
    if handle:
        load().svr2_destroy(handle)
