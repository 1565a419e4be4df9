"""ctypes binding of the C ABI in include/mwa_b200.h (libmwa_b200.so, built in-tree by build.py).

There is no fallback: if the library is missing or a call returns a non-zero status, a Python
exception is raised.  Tensors cross the boundary as raw device pointers + sizes; the stream is
torch's current CUDA stream.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int32, c_int64, c_void_p, POINTER

import torch

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "libmwa_b200.so")

MWA_OK = 0
ALGO_AUTO, ALGO_SIMT, ALGO_TCGEN05 = 0, 1, 2
ABI_VERSION = 1

# name -> (restype, argtypes); mirrors include/mwa_b200.h one to one
_SIGNATURES = {
    "mwa_b200_abi_version": (c_int, []),
    "mwa_b200_status_string": (c_char_p, [c_int]),
    "mwa_b200_last_cuda_error": (c_char_p, []),
    "gdn_param_bytes": (c_int64, [c_int]),
    "gdn_prepare": (c_int, [c_void_p, c_void_p, c_int, c_float, c_float, c_float, c_void_p, c_int64, c_void_p]),
    "gdn_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int64, c_int, c_int, c_int, c_void_p]),
    "gdn_forward_planes": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int64, c_int, c_int, c_int, c_int,
                                   c_void_p]),
    "gdn_backward_workspace_bytes": (c_int64, [c_int64, c_int, c_int64]),
    "gdn_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_float, c_void_p, c_void_p,
                             c_void_p, c_void_p, c_int64, c_int64, c_int, c_int64, c_int, c_int, c_void_p]),
    "gdn_param_offset": (c_int64, [c_int, c_int]),
    "gdn_bwd_square": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "gdn_bwd_dn": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int64, c_int, c_int,
                           c_void_p]),
    "gdn_bwd_dx": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "gdn_bwd_finalize": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_float, c_void_p, c_void_p,
                                 c_void_p, c_int64, c_int, c_int64, c_int, c_void_p]),
    "mwa_param_bytes": (c_int64, [c_int, c_int, c_int]),
    "mwa_prepare": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float,
                            c_void_p, c_int64, c_void_p]),
    "mwa_debug_set_timing_buffer": (None, [c_void_p]),
    "mwa_workspace_bytes": (c_int64, [c_int, c_int, c_int, c_int]),
    "mwa_fast_path_needs_nchw": (c_int, [c_int, c_int, c_int]),
    "conv_image_bytes": (c_int64, [c_int, c_int, c_int, c_int, c_int]),
    "conv_split_bytes": (c_int64, [c_int, c_int, c_int, c_int]),
    "conv_prepare": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int64, c_void_p]),
    "conv_forward": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int,
                             c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "gemm_tokens_forward": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p]),
    "conv_act_split": (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "conv_forward_ex": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int64,
                                c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p,
                                c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "mwa_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                            c_int, c_int, c_void_p, c_void_p, c_int64, c_void_p]),
    "window_attention_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_int,
                                         c_void_p]),
    "mwa_backward": (c_int, [c_void_p] * 12 + [c_int] * 8 + [c_void_p]),
    "window_attention_backward": (c_int, [c_void_p] * 10 + [c_int64, c_int, c_int, c_int, c_int, c_void_p]),
    "mwa_bwd_gather": (c_int, [c_void_p] * 6 + [c_int] * 7 + [c_void_p]),
    "mwa_bwd_core": (c_int, [c_void_p] * 8 + [c_int64] + [c_int] * 7 + [c_void_p]),
    "mwa_bwd_scatter": (c_int, [c_void_p] * 3 + [c_int] * 7 + [c_void_p]),
    "gate_residual_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "gate_residual_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "round_ste_forward": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_void_p]),
    "quantize_offset_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_int64,
                                        c_int, c_int64, c_void_p]),
    "lrp_add_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_int64, c_void_p]),
    "quantize_levels_forward": (c_int, [c_void_p, c_void_p, c_int64, c_float, c_void_p]),
    "alpha_pyramid_level_offset": (c_int64, [c_int, c_int, c_int, c_int]),
    "alpha_pyramid_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "ms_ssim_level_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p,
                                      c_void_p]),
    "ms_ssim_pool_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                     c_void_p]),
    "ms_ssim_level_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "rans_encode_with_indexes": (c_int64, [c_void_p, c_void_p, c_int64, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p,
                                           c_int64]),
    "rans_decode_with_indexes": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_int, c_void_p, c_void_p,
                                         c_int, c_void_p]),
    "rans_lanes_encode": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int,
                                  c_void_p, c_int64, c_void_p, c_void_p]),
    "rans_lanes_pack": (c_int, [c_void_p, c_int64, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "rans_lanes_decode": (c_int, [c_void_p, c_int64, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int64, c_int64, c_void_p,
                                  c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "rate_workspace_bytes": (c_int64, [c_int]),
    "rate_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int64,
                             c_void_p, c_void_p, c_int, c_int64, c_void_p, c_int64, c_void_p, c_void_p]),
    "mask_constraint_forward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "rgba8_ingest": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "rgba8_egress": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None

# kernel launches issued through this binding (bench.py's `gpu_launches`): the wrappers add what each call launches
launch_count = 0


def count_launches(n: int) -> None:
    global launch_count
    launch_count += n


class MwaB200Error(RuntimeError):
    pass


def load() -> ctypes.CDLL:
    """dlopen the in-tree library and type its entry points.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MwaB200Error(
            f"{LIB_PATH} not found: build it with `python __graft_entry__.py build` "
            "(nvcc, sm_100a).  This package has no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the header and the library drifted apart
        fn.restype = res
        fn.argtypes = args
    got = lib.mwa_b200_abi_version()
    if got != ABI_VERSION:
        raise MwaB200Error(f"ABI version mismatch: library {got}, binding {ABI_VERSION}")
    _lib = lib
    return lib


def check(status: int, what: str) -> None:
    if status == MWA_OK:
        return
    lib = load()
    msg = lib.mwa_b200_status_string(status).decode()
    extra = lib.mwa_b200_last_cuda_error().decode() if status == -5 else ""
    raise MwaB200Error(f"{what} failed: {msg} (status {status}) {extra}".rstrip())


def ptr(t: torch.Tensor | None):
    return None if t is None else t.data_ptr()


def stream_handle() -> int:
    return torch.cuda.current_stream().cuda_stream


def require_cuda_f32(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise MwaB200Error(f"{name} must be a CUDA tensor (got {t.device}); this package is sm_100a-only "
                           "and has no CPU fallback")
    if t.dtype != torch.float32:
        raise MwaB200Error(f"{name} must be float32 (got {t.dtype})")


# Opt-in (default OFF: the reference's gradients are fp32 end to end).  MWA_B200_WGRAD_TF32=1 in the environment, or
# `mwa_b200._abi.WGRAD_TF32 = True`, lets the LARGE-K parameter-gradient GEMMs use TF32 products (see tf32_reduction).
WGRAD_TF32 = os.environ.get("MWA_B200_WGRAD_TF32", "0") == "1"


class tf32_reduction:
    """Context for the LARGE-K parameter-gradient GEMMs of the backward (dW = dY^T X over all tokens, dgamma = dn (x^2)^T
    over all pixels: K = 10^4 ... 10^6).  A no-op unless WGRAD_TF32 was switched on explicitly: then the library GEMM
    may use TF32 tensor-core products with fp32 accumulation (a 2^-11 relative error per product averages out over that
    many terms, observed ~1e-5 relative on the sums; the fp32 SIMT SGEMM these shapes otherwise fall to is 27 % of the
    training step).  The switch it flips, `torch.backends.cuda.matmul.allow_tf32`, is process-global: with it on, a
    matmul running concurrently on another thread can pick up TF32 too -- which is why this is opt-in.  The per-pixel /
    per-token contractions (K = C) always stay in full fp32."""

    MIN_K = 8192        # below this the averaging argument is weak and the fp32 GEMM is cheap anyway

    def __init__(self, k: int):
        self.on = WGRAD_TF32 and k >= self.MIN_K

    def __enter__(self):
        if self.on:
            self.prev = torch.backends.cuda.matmul.allow_tf32
            torch.backends.cuda.matmul.allow_tf32 = True

    def __exit__(self, *exc):
        if self.on:
            torch.backends.cuda.matmul.allow_tf32 = self.prev
        return False
