"""ctypes loader for the C-ABI library (include/rsn_b200.h).  There is no CPU fallback: every op fails
loudly if the library is missing or the device is not a B200.

`lib()` / `call()` = the product library librsn_b200.so.  `lib_dbg()` / `call_dbg()` = the test build
librsn_b200_dbg.so (include/rsn_b200_test.h: environment switches, probes, the one-launch backward), loaded only
when a test or an experiment script asks for it."""
from __future__ import annotations

import ctypes
import os
from ctypes import c_double, c_float, c_int, c_int64, c_longlong, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RSN_B200_LIB") or os.path.join(_HERE, "librsn_b200.so")   # env override: kernel experiments
LIB_DBG_PATH = os.environ.get("RSN_B200_LIB_DBG") or os.path.join(_HERE, "librsn_b200_dbg.so")
_lib = None
_lib_dbg = None

P, I64, I32, F32, F64, LL = c_void_p, c_int64, c_int, c_float, c_double, c_longlong
_SIGNATURES = {
    "rsn_version": ([], c_int),
    "rsn_last_error": ([], ctypes.c_char_p),
    "rsn_device_ok": ([], c_int),
    "rsn_sample_spaced": ([P, P, P, P, I64, I32, F32, P, P, I64, I64, P, P], c_int),
    "rsn_pdf_resample": ([P, I64, P, P, P, P, P, I32, F32, F32, P, P, P, I64, I64, I64, P, P], c_int),
    "rsn_render_weights": ([P, P, I64, P, P, I64, P, P, P, I64, I64, P], c_int),
    "rsn_ipe_encode": ([P, P, P, I64, P], c_int),
    "rsn_ide_encode": ([P, P, P, I64, P], c_int),
    "rsn_composite_fwd": ([P, P, P, I64, P, I64, P, P, P, P, I64, I64, P, P], c_int),
    "rsn_composite_bwd": ([P, P, P, I64, P, I64, P, P, P, P, P, I64, I64, P, P], c_int),
    "rsn_composite16_fwd": ([P, P, P, I64, P, P, P, P, P, P, P, P, P, I64, I64, P, P], c_int),
    "rsn_composite16_bwd": ([P, P, P, I64, P, P, P, P, P, P, P, P, P, P, P, P, I64, I64, P, P], c_int),
    "rsn_field_forward": ([P, P, I32, P, P, P, P, I64, I64, P, P, P, P], c_int),
    "rsn_field_forward_train": ([P, P, I32, P, P, P, P, I64, I64, P, P, P, P, P, P], c_int),
    "rsn_field_forward_points": ([P, P, P, P, P, P, I64, P, P, P, P], c_int),
    "rsn_frustum_gaussians": ([P, P, P, P, I64, I64, P, P, P], c_int),
    "rsn_contract": ([P, P, P, P, I64, P], c_int),
    "rsn_field_stash_bytes": ([I64], c_int64),
    "rsn_field_normals": ([P, P, P, I64, I64, P, P], c_int),
    "rsn_field_blob_t_bytes": ([], c_int64),
    "rsn_field_backward": ([P, P, I32, P, P, P, P, I64, I64, P, P, P, P, P, P, P, P], c_int),
    "rsn_field_dy_stash_bytes": ([I64], c_int64),
    "rsn_field_wgrad": ([P, P, I64, P, P, P, I64, P], c_int),
    "rsn_field_wgrad_workspace_bytes": ([], c_int64),
    "rsn_field_wgrad_layout": ([P, P, P], c_int),
    "rsn_field_wgrad_finish": ([P, P, P, P, P], c_int),
    "rsn_unpack_grads": ([P, P, P], c_int),
    "rsn_field_flat_layout": ([P], c_int64),
    "rsn_pack_field": ([P, P, P, P, P, P], c_int),
    "rsn_field_blob_bytes": ([], c_int64),
    "rsn_field_bias_count": ([], c_int64),
    "rsn_ipe_freqs": ([P], c_int),
    "rsn_radam_step": ([P, P, P, P, P, P, P, F64, F64, LL, F64, F64, F64, F32, P], c_int),
    "rsn_loss_workspace_bytes": ([], c_int64),
    "rsn_loss_fwd": ([P] * 12 + [I64, P], c_int),
    "rsn_loss_bwd": ([P] * 16 + [I64, P], c_int),
    "rsn_reflect_setup": ([P, P, P, P, P, I32, P, P, P, P, P, P, P, I64, P], c_int),
    "rsn_reflect_compact": ([P, P, P, P, I64, P], c_int),
    "rsn_reflect_bundle_fwd": ([P, P, P, P, P, P, P, P, P, P, I64, P], c_int),
    "rsn_reflect_bundle_bwd": ([P, P, P, P, P, P, I64, P], c_int),
    "rsn_reflect_compose_fwd": ([P, P, P, P, P, I64, P, P, I32, P, P, P, I64, P], c_int),
    "rsn_reflect_compose_bwd": ([P, P, P, P, P, I64, P, P, P, P, P, I64, P], c_int),
    "rsn_raygen": ([P, P, P, P, P, I64, I64, I64, I64, P, P, P, P, P, I64, P], c_int),
}
# include/rsn_b200_test.h: the test build exports everything above plus these
_SIGNATURES_DBG = {
    "rsn_debug_fwd_trace": ([P, I32], c_int),
    "rsn_probe_umma_kmajor": ([P, P, I64, I64, I64, P, P], c_int),
    "rsn_probe_umma_2cta": ([P, P, I64, I64, P, P], c_int),
    "rsn_probe_epilogue": ([I64, I64, I64, P, P], c_int),
    "rsn_probe_tmem_rate": ([I64, I64, I64, I64, P, P], c_int),
    "rsn_probe_umma_ts": ([P, P, I64, I64, P, I64, P, P], c_int),
    "rsn_probe_umma_rate_2cta": ([I64, I64, I64, P, P], c_int),
    "rsn_probe_umma_rate": ([I32, I32, I64, I64, P, P], c_int),
    "rsn_probe_umma_mnmajor": ([P, P, I64, I64, P, P], c_int),
    "rsn_probe_umma_mnmajor_cm": ([P, P, I64, I64, I64, P, I64, P, P], c_int),
}


def _load(path: str, signatures) -> ctypes.CDLL:
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} is missing: build it with `python -m reflect_sampling_nerf_b200.build` "
            "(there is no CPU or PyTorch fallback for the rsn_b200 kernels)")
    handle = ctypes.CDLL(path)
    for name, (argtypes, restype) in signatures.items():
        fn = getattr(handle, name)
        fn.argtypes = argtypes
        fn.restype = restype
    return handle


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        _lib = _load(LIB_PATH, _SIGNATURES)
    return _lib


def lib_dbg() -> ctypes.CDLL:
    global _lib_dbg
    if _lib_dbg is None:
        _lib_dbg = _load(LIB_DBG_PATH, {**_SIGNATURES, **_SIGNATURES_DBG})
    return _lib_dbg


# `use_dbg(True)` routes call() through the test build (tests of the alternative kernel forms); default: the product.
_active = lib


def use_dbg(on: bool) -> None:
    global _active
    _active = lib_dbg if on else lib


def active() -> ctypes.CDLL:
    return _active()


def call(name: str, *args) -> None:
    handle = _active()
    code = getattr(handle, name)(*args)
    if code != 0:
        raise RuntimeError(f"{name} failed with code {code}: {handle.rsn_last_error().decode()}")


def ptr(t):
    """Device pointer of a (contiguous-as-needed) CUDA tensor, or NULL for None."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("rsn_b200 ops need CUDA tensors (no CPU fallback)")
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream
