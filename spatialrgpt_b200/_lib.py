"""ctypes binding of libsrgpt_b200.so (the C-ABI declared in include/srgpt_b200.h).

There is deliberately NO fallback: if the shared library cannot be built/loaded, or a kernel
returns an error, a ``SrgptError`` is raised.  Nothing in this package computes on the CPU or
through torch operators on the product path.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

from . import _build

_lock = threading.Lock()
_libs = {}       # element type ("bf16" / "f16") -> typed CDLL
_elem = "bf16"   # element type whose library load() returns; switched by ops.elem_dtype() around a model's calls


class SrgptError(RuntimeError):
    pass


vp, ci, cf, cll = C.c_void_p, C.c_int, C.c_float, C.c_longlong

# name -> (restype, argtypes); mirrors include/srgpt_b200.h one to one
SIGNATURES = {
    "srgpt_abi_version": (ci, []),
    "srgpt_elem_type": (ci, []),
    "srgpt_last_error": (C.c_char_p, []),
    "srgpt_device_info": (ci, [C.POINTER(ci), C.POINTER(ci), C.POINTER(ci)]),
    "srgpt_trace_begin": (ci, [vp, ci]),
    "srgpt_trace_end": (ci, []),
    "srgpt_gemm_workspace_bytes": (cll, []),
    "srgpt_gemm_set_workspace": (ci, [vp, cll]),
    "srgpt_gemm_bf16": (ci, [vp, ci, vp, ci, vp, ci, ci, ci, ci, vp, vp, ci, ci, ci, ci, vp]),
    "srgpt_layernorm_bf16": (ci, [vp, ci, vp, vp, vp, ci, ci, ci, cf, ci, vp]),
    "srgpt_downsample_layernorm_bf16": (ci, [vp, vp, vp, vp, ci, ci, ci, cf, vp]),
    "srgpt_rmsnorm_bf16": (ci, [vp, ci, vp, vp, ci, ci, ci, cf, vp]),
    "srgpt_patchify_bf16": (ci, [vp, ci, vp, ci, ci, ci, ci, vp]),
    "srgpt_clip_embed_bf16": (ci, [vp, vp, vp, vp, ci, ci, ci, vp]),
    "srgpt_splice_rows_bf16": (ci, [vp, vp, vp, vp, vp, vp, vp, ci, ci, vp]),
    "srgpt_mask_weights_workspace": (cll, [ci, ci, ci]),
    "srgpt_mask_weights": (ci, [vp, ci, vp, vp, ci, ci, ci, ci, ci, cf, ci, vp]),
    "srgpt_mask_pool_workspace": (cll, [ci, ci, ci, ci]),
    "srgpt_mask_pool_bf16": (ci, [vp, vp, vp, vp, ci, ci, ci, ci, vp]),
    "srgpt_adaptive_avgpool_bf16": (ci, [vp, vp, ci, ci, ci, ci, ci, vp]),
    "srgpt_reorder_rows_bf16": (ci, [vp, vp, ci, ci, ci, ci, ci, vp]),
    "srgpt_depth_to_u8x3": (ci, [vp, ci, ci, vp, ci, ci, vp, vp]),
    "srgpt_attention_prefill_bf16": (ci, [vp, vp, vp, vp, ci, ci, ci, ci, ci, ci, ci, ci, cf, ci, vp]),
    "srgpt_attention_prefill_varlen_bf16": (ci, [vp, vp, vp, vp, ci, ci, ci, ci, vp, ci, ci, ci, ci, ci, cf, ci, vp]),
    "srgpt_rope_kv_append_bf16": (ci, [vp, ci, ci, ci, ci, vp, vp, vp, vp, vp, ci, vp]),
    "srgpt_rope_kv_append_varlen_bf16": (ci, [vp, ci, ci, ci, ci, vp, vp, vp, vp, vp, ci, ci, ci, vp, vp]),
    "srgpt_attention_prefill_paged_workspace": (cll, [ci, ci, ci, ci, ci]),
    "srgpt_attention_prefill_paged_bf16": (ci, [vp, ci, vp, ci, vp, vp, ci, ci, ci, vp, vp, ci, ci, ci, ci, ci, cf, vp, cll, vp]),
    "srgpt_attention_decode_bf16": (ci, [vp, vp, vp, vp, ci, vp, ci, ci, ci, cf, vp]),
    "srgpt_gemv_bf16": (ci, [vp, vp, ci, vp, ci, ci, vp, cf, vp, ci, ci, ci, ci, vp, vp, vp, vp, vp, ci, vp]),
    "srgpt_lm_head_workspace": (cll, [ci]),
    "srgpt_lm_head_argmax_bf16": (ci, [vp, vp, ci, ci, ci, vp, cf, vp, vp, vp, vp, vp, vp, vp, vp]),
    "srgpt_argmax_f32": (ci, [vp, ci, ci, vp, vp]),
    "srgpt_argmax_bf16": (ci, [vp, ci, ci, ci, vp, vp]),
    "srgpt_beam_candidates_bf16": (ci, [vp, ci, ci, ci, vp, ci, vp, vp, vp]),
    "srgpt_sample_top_p_f32": (ci, [vp, ci, vp, vp, vp, ci, vp, vp, vp, ci, vp]),
    "srgpt_resample_u8": (ci, [vp, vp, ci, ci, ci, ci, ci, vp, vp, ci, vp]),
    "srgpt_u8_to_normalized_chw": (ci, [vp, vp, ci, ci, ci, C.c_double, vp, vp, ci, vp]),
    "srgpt_resize_nearest_u8": (ci, [vp, vp, ci, ci, ci, ci, vp, vp, vp]),
    "srgpt_attention_decode_batched_bf16": (ci, [vp, ci, vp, ci, vp, vp, ci, ci, vp, ci, ci, ci, ci, cf, vp]),
    "srgpt_decode_batch_advance": (ci, [vp, vp, vp, ci, vp, vp, vp, ci, vp, vp]),
    "srgpt_gemv_tp_bf16": (ci, [vp, vp, ci, vp, ci, ci, vp, cf, ci, ci, ci, ci, vp, vp, vp, vp, vp, ci, ci, ci, vp, vp]),
    "srgpt_attention_decode_tp_bf16": (ci, [vp, vp, vp, vp, ci, vp, ci, ci, ci, ci, ci, cf, vp]),
    "srgpt_tp_residual_add_bf16": (ci, [vp, vp, ci, vp]),
    "srgpt_lm_head_local_best_bf16": (ci, [vp, vp, ci, ci, ci, vp, cf, vp, ci, vp, vp]),
    "srgpt_tp_pick_token": (ci, [vp, ci, vp, vp, ci, vp, vp, vp, vp]),
    "srgpt_tp_comm_bytes": (cll, [ci, ci, ci]),
    "srgpt_tp_comm_slot_offset": (cll, [ci, ci, ci]),
    "srgpt_tp_allreduce_residual_bf16": (ci, [vp, ci, ci, cll, ci, vp, vp, vp, ci, vp]),
    "srgpt_tp_allgather_pick_token": (ci, [vp, ci, ci, cll, ci, vp, vp, vp, ci, vp, vp, vp, vp]),
    "srgpt_siglip_layers_bf16": (ci, [vp, vp, ci, vp, vp, vp, vp, ci, ci, ci, ci, ci, cf, vp]),
    "srgpt_vit_layers_bf16": (ci, [vp, vp, ci, vp, vp, vp, vp, ci, ci, ci, ci, ci, cf, ci, vp]),
    "srgpt_llama_prefill_layers_bf16": (ci, [vp, vp, ci, vp, vp, vp, vp, ci, ci, ci, ci, ci, ci, cf, vp, vp, vp, vp, ci, ci, vp, ci, ci, vp]),
    "srgpt_llama_prefill_layers_paged_bf16": (ci, [vp, vp, ci, vp, vp, vp, vp, vp, cll, ci, ci, ci, ci, ci, ci, cf, vp, vp, vp, vp, ci, ci, ci,
                                                   vp, ci, ci, vp]),
    "srgpt_llama_decode_step_bf16": (ci, [vp, vp, ci, vp, vp, vp, ci, ci, ci, ci, ci, cf, vp, vp, vp, vp, ci, vp, vp, ci, vp, vp, vp, vp,
                                          vp, vp]),
}


class SiglipLayerWeights(C.Structure):
    _fields_ = [(n, vp) for n in ("ln1_w", "ln1_b", "qkv_w", "qkv_b", "out_w", "out_b", "ln2_w", "ln2_b", "fc1_w", "fc1_b", "fc2_w", "fc2_b")]


class LlamaLayerWeights(C.Structure):
    _fields_ = [(n, vp) for n in ("in_norm", "qkv_w", "o_w", "post_norm", "gateup_w", "down_w", "kv_pages")]


def lib_path(elem: str = "bf16") -> str:
    return _build.VARIANTS[elem][0]


def current_elem() -> str:
    return _elem


def set_elem(elem: str) -> str:
    """Selects which build of the library (bf16 or f16 elements) ``load()`` hands out; returns the previous setting."""
    global _elem
    if elem not in _build.VARIANTS:
        raise SrgptError(f"unsupported element type {elem!r} (have {sorted(_build.VARIANTS)})")
    prev, _elem = _elem, elem
    return prev


def load(build_if_missing: bool = True, elem: str = None):
    """Load (building first if the .so is missing/stale and nvcc is present) and type the library of the given (default: the
    current) element type."""
    elem = elem or _elem
    with _lock:
        if elem in _libs:
            return _libs[elem]
        path = lib_path(elem)
        if build_if_missing and _build.is_stale():
            try:
                _build.build(verbose=False)
            except Exception as e:  # stale-but-present is still loadable; missing is fatal
                if not os.path.exists(path):
                    raise SrgptError(f"{os.path.basename(path)} is missing and could not be built: {e}") from e
        if not os.path.exists(path):
            raise SrgptError(f"{path} not found; run `python -c 'import __graft_entry__ as g; g.build()'`")
        try:
            import torch  # noqa: F401  (loads libcudart.so.12 that the library links against)
        except Exception:
            pass
        lib = C.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            try:
                fn = getattr(lib, name)
            except AttributeError as e:
                raise SrgptError(f"{path} does not export {name}") from e
            fn.restype = res
            fn.argtypes = args
        if lib.srgpt_abi_version() != 1:
            raise SrgptError(f"ABI version mismatch between _lib.py and {os.path.basename(path)}")
        if lib.srgpt_elem_type() != {"bf16": 0, "f16": 1}[elem]:
            raise SrgptError(f"{path} was not built for {elem} elements")
        _libs[elem] = lib
        return lib


def last_error() -> str:
    return (load().srgpt_last_error() or b"").decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise SrgptError(f"{what} failed with code {rc}: {last_error()}")


def device_info():
    sm, maj, mnr = ci(0), ci(0), ci(0)
    check(load().srgpt_device_info(C.byref(sm), C.byref(maj), C.byref(mnr)), "srgpt_device_info")
    return sm.value, maj.value, mnr.value
