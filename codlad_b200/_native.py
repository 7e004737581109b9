"""ctypes binding of libcodlad_b200.so (C ABI: include/codlad_b200.h).

There is NO fallback: if the library is missing or does not load, every entry point raises.
Build it with `python -m codlad_b200.build` (or `__graft_entry__.build()`).
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CB2_LIB") or os.path.join(_HERE, "libcodlad_b200.so")      # CB2_LIB: experiment builds
ABI_VERSION = 4

PRECISION = {"fp32": 0, "f32": 0, "f16": 1, "fp16": 1}


class cb2_tensor(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("numel", C.c_longlong)]


# name -> (restype, argtypes); this table is also what tests/test_cabi.py checks against the header
_P, _I, _LL = C.c_void_p, C.c_int, C.c_longlong
SIGNATURES = {
    "cb2_abi_version": (_I, []),
    "cb2_last_error": (C.c_char_p, []),
    "cb2_denoiser_create": (_I, [C.POINTER(cb2_tensor), _I, _P, _I, C.POINTER(_P)]),
    "cb2_denoiser_destroy": (None, [_P]),
    "cb2_vae_create": (_I, [C.POINTER(cb2_tensor), _I, _P, _P, _I, C.POINTER(_P)]),
    "cb2_vae_destroy": (None, [_P]),
    "cb2_plan_create": (_I, [_P, _I, _I, _I, _I, _I, C.POINTER(_P)]),
    "cb2_plan_destroy": (None, [_P]),
    "cb2_plan_K": (_I, [_P]),
    "cb2_plan_launches": (_LL, [_P]),
    "cb2_plan_set_frames": (_I, [_P, _P, _P, _P, _P, _P]),
    "cb2_plan_forward": (_I, [_P, _P, _P, _P, _P]),
    "cb2_plan_forward_partial": (_I, [_P, _P, _P, _I, _P]),
    "cb2_plan_set_schedule": (_I, [_P, _P, _P, _I, _P]),
    "cb2_plan_set_ddim_schedule": (_I, [_P, _P, _P, _I, _P]),
    "cb2_plan_sample": (_I, [_P, _P, _P, _I, _P]),
    "cb2_plan_set_inpaint": (_I, [_P, _P, _P, _P, _I, _P]),
    "cb2_plan_set_topology": (_I, [_P, _P, _P, _P, _P, _I, _P, _P, _P, _P]),
    "cb2_plan_decode": (_I, [_P, _P, _P, _I, _P, _P, _P, _P, _P]),
    "cb2_plan_residue_clashes": (_I, [_P, _P, C.c_float, _I, _P, _P, _P]),
    "cb2_plan_buffer": (_I, [_P, C.c_char_p, _P, _LL, _P]),
    "cb2_plan_run_edge_kernel": (_I, [_P, _I, _I, _P]),
    "cb2_plan_run_stage": (_I, [_P, _P, _I, _I, _P, _P]),
    "cb2_knn_topk": (_I, [_P, _P, _I, _I, _I, _P, _P, _P]),
    "cb2_vq_lookup": (_I, [_P, _P, _I, _I, _P, _P, _I, _P, _P, _P]),
    "cb2_p_sample": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _P, _P]),
    "cb2_ddim_sample": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _P, _P]),
    "cb2_ic_to_xyz": (_I, [_P, _P, _I, _I, _P, _P, _P, _P, _P, _P, _P]),
    "cb2_superposed_rmsd": (_I, [_P, _P, _P, _I, _P, _P]),
    "cb2_eval_bond_graphs": (_I, [_P, _P, _P, _P, _I, _I, _P, _I, C.c_float, _P, _P, _P]),
    "cb2_pair_losses": (_I, [_P, _P, _P, _I, C.c_longlong, C.c_float, C.c_float, _P, _P]),
    "cb2_keys_once": (_I, [_P, C.c_longlong, _P, _P]),
}

# include/codlad_b200_train.h (the train_latent step, SURVEY.md section 8 row f-1)
_F = C.c_float
SIGNATURES.update({
    "cb2t_gemm": (_I, [_P, _P, _P, _I, _I, _I, _LL, _LL, _LL, _I, _I, _I, _P]),
    "cb2t_set_gemm_mode": (_I, [_I]),
    "cb2t_bias_gelu_fwd": (_I, [_P, _P, _LL, _I, _P, _P]),
    "cb2t_linear_bias_gelu_fwd": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _LL, _LL, _LL, _P]),
    "cb2t_gelu_bwd": (_I, [_P, _P, _LL, _P, _P]),
    "cb2t_gelu_bwd_colsum": (_I, [_P, _P, _LL, _I, _P, _P, _I, _P]),
    "cb2t_elementwise": (_I, [_I, _P, _P, _F, _LL, _P, _P]),
    "cb2t_edge_combine_gelu_fwd": (_I, [_P, _P, _P, _P, _P, _I, _LL, _P, _P]),
    "cb2t_edge_gather_bwd": (_I, [_P, _I, _I, _P, _P, _P, _P, _P]),
    "cb2t_masked_sum_fwd": (_I, [_P, _P, _I, _I, _F, _P, _P]),
    "cb2t_masked_sum_bwd": (_I, [_P, _P, _I, _LL, _F, _P, _P]),
    "cb2t_ln_mod_fwd": (_I, [_P, _P, _P, _LL, _LL, _P, _P, _P, _LL, _P, _F, _P, _P, _P, _P]),
    "cb2t_ln_mod_bwd": (_I, [_P, _P, _P, _LL, _LL, _P, _P, _P, _LL, _P, _P, _P, _P, _P, _I, _P]),
    "cb2t_edge_raw_features": (_I, [_P, _P, _P, _I, _I, _I, _P, _P]),
    "cb2t_row_gather_add": (_I, [_P, _P, _P, _LL, _P]),
    "cb2t_index_sum": (_I, [_P, _P, _LL, _I, _I, _P, _I, _P]),
    "cb2t_colsum": (_I, [_P, _LL, _I, _LL, _P, _I, _P]),
    "cb2t_sumsq": (_I, [_P, _LL, _P, _P]),
    "cb2t_adamw_ema": (_I, [_P, _P, _P, _P, _P, _LL, _F, _F, _F, _F, _F, _I, _F, _P, _F, _P]),
})

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: the CUDA library has not been built. Run `python -m codlad_b200.build`. "
                "codlad_b200 has no CPU or PyTorch fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)       # AttributeError if the export is missing
            fn.restype = res
            fn.argtypes = args
        if handle.cb2_abi_version() != ABI_VERSION:
            raise RuntimeError(f"libcodlad_b200 ABI {handle.cb2_abi_version()} != binding ABI {ABI_VERSION}; rebuild")
        _lib = handle
    return _lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().cb2_last_error()
        raise RuntimeError(f"codlad_b200 {what} failed (code {rc}): {msg.decode() if msg else ''}")


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("codlad_b200 needs a CUDA device (sm_100a); there is no CPU fallback")


def dptr(t: torch.Tensor, dtype=None) -> int:
    """Device pointer of a contiguous CUDA tensor (borrowed for the duration of the call)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise ValueError("expected a CUDA tensor")
    if not t.is_contiguous():
        raise ValueError("expected a contiguous tensor")
    if dtype is not None and t.dtype != dtype:
        raise ValueError(f"expected dtype {dtype}, got {t.dtype}")
    return t.data_ptr()


def hptr(t: torch.Tensor, dtype) -> int:
    if t.is_cuda or not t.is_contiguous() or t.dtype != dtype:
        raise ValueError(f"expected a contiguous CPU tensor of dtype {dtype}")
    return t.data_ptr()


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def tensor_table(state: dict):
    """state_dict -> (cb2_tensor array, keepalive list).  Tensors are staged as contiguous CPU fp32."""
    keep, rows = [], []
    for name, t in state.items():
        if not torch.is_tensor(t) or not t.dtype.is_floating_point:
            continue
        h = t.detach().to(device="cpu", dtype=torch.float32).contiguous()
        keep.append(h)
        rows.append(cb2_tensor(name.encode(), h.data_ptr(), h.numel()))
    arr = (cb2_tensor * len(rows))(*rows)
    return arr, keep
