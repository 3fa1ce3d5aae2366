"""ctypes binding of liblfi_b200.so (the C ABI declared in include/lfi_b200.h).

This is the *only* place the shared library is touched.  There is no fallback: if the library is
missing, or a call returns a non-zero status, a RuntimeError is raised (the reference's error
convention is Python exceptions/asserts, SURVEY.md §8(b)).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "liblfi_b200.so")
NMOD = 4
ABI_VERSION = 6

GEMM_FP32, GEMM_BF16X3, GEMM_BF16 = 0, 1, 2
EPI_BIAS, EPI_LRELU, EPI_ACCUM, EPI_LRELU_BWD = 1, 2, 4, 8

_fp = C.POINTER(C.c_float)


class Shape(C.Structure):
    _fields_ = [
        ("C", C.c_int32), ("K", C.c_int32), ("H", C.c_int32), ("D", C.c_int32), ("G", C.c_int32),
        ("affine", C.c_int32), ("scale_eps", C.c_float),
        ("hist", C.c_int32 * NMOD), ("dim", C.c_int32 * NMOD), ("ehid", C.c_int32 * NMOD),
        ("f_raw", C.c_int32),
    ]


class Params(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in
                ("an_bias", "an_logs", "w", "wc", "bc", "w_ih", "b_ih", "w_hh", "b_hh", "wf", "bf", "lf")] + [
        ("enc_w_ih", C.c_void_p * NMOD), ("enc_w_hh", C.c_void_p * NMOD),
        ("enc_b_ih", C.c_void_p * NMOD), ("enc_b_hh", C.c_void_p * NMOD),
    ]


class FseqShape(C.Structure):
    _fields_ = [("In", C.c_int32), ("Out", C.c_int32), ("H", C.c_int32), ("D", C.c_int32), ("F", C.c_int32), ("G", C.c_int32),
                ("logscale_factor", C.c_float)]


FSEQ_PARAMS = ("wc", "bc", "w_ih", "b_ih", "w_hh", "b_hh", "wf", "bf", "lf")


class FseqParams(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in FSEQ_PARAMS]


class Batch(C.Structure):
    _fields_ = [("x", C.c_void_p * NMOD), ("mask", C.c_void_p * NMOD), ("B", C.c_int32), ("T", C.c_int32)]


# name -> (restype, argtypes); every symbol include/lfi_b200.h declares
_P, _SZ, _I, _F, _L = C.c_void_p, C.c_size_t, C.c_int, C.c_float, C.c_long
_SH, _PR, _BT = C.POINTER(Shape), C.POINTER(Params), C.POINTER(Batch)
_FS, _FP = C.POINTER(FseqShape), C.POINTER(FseqParams)
SYMBOLS = {
    "lfi_last_error": (C.c_char_p, []),
    "lfi_abi_version": (_I, []),
    "lfi_launch_count": (_L, []),
    "lfi_set_grad_ready_event": (_I, [_P]),
    "lfi_set_derived_ready_event": (_I, [_P]),
    "lfi_expand_faces": (_I, [_P, _P, _P, _SZ, _I, _I, _I, _P, _P]),
    "lfi_feature_dim": (_I, [_SH]),
    "lfi_feature_dim_folded": (_I, [_SH]),
    "lfi_start_ts": (_I, [_SH]),
    "lfi_coupling_out": (_I, [_SH]),
    "lfi_derived_bytes": (_SZ, [_SH]),
    "lfi_train_ws_bytes": (_SZ, [_SH, _I, _I, _I]),
    "lfi_sample_ws_bytes": (_SZ, [_SH, _I, _I, _I, _I]),
    "lfi_invconv_ws_bytes": (_SZ, [_I, _I]),
    "lfi_gemm_ws_bytes": (_SZ, [_I, _I, _I, _I, _I, _I, _I]),
    "lfi_feature_ws_bytes": (_SZ, [_SH, _I, _I, _I, _I]),
    "lfi_flowstep_ws_bytes": (_SZ, [_SH, _I]),
    "lfi_flowstep_stash_bytes": (_SZ, [_SH, _I]),
    "lfi_flowstep_bwd_ws_bytes": (_SZ, [_SH, _I]),
    "lfi_flowstep_fwd_train": (_I, [_SH, _P, _PR, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _P, _SZ, _P, _SZ, _P]),
    "lfi_flowstep_bwd": (_I, [_SH, _P, _PR, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _PR, _I, _P, _SZ, _P, _SZ, _P]),
    "lfi_derive": (_I, [_SH, _PR, _P, _P, _I, _P]),
    "lfi_invconv_compose": (_I, [_I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "lfi_invconv_compose_bwd": (_I, [_I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "lfi_seq_train_fwd": (_I, [_SH, _P, _PR, _BT, _P, _P, _P, _P, _SZ, _I, _P]),
    "lfi_seq_train_bwd": (_I, [_SH, _P, _PR, _BT, _P, _P, _PR, _P, _SZ, _I, _P]),
    "lfi_seq_sample": (_I, [_SH, _P, _PR, _BT, _I, _P, _P, _P, _I, _I, _P, _SZ, _I, _P]),
    "lfi_feature_encode": (_I, [_SH, _PR, _BT, _I, _I, _P, _P, _SZ, _I, _P]),
    "lfi_flowstep": (_I, [_SH, _P, _PR, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _P, _SZ, _P]),
    "lfi_actnorm": (_I, [_P, _P, _P, _P, _I, _I, _I, _P]),
    "lfi_matmul": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "lfi_nll": (_I, [_P, _P, _P, _I, _I, _P]),
    "lfi_actnorm_bwd": (_I, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P]),
    "lfi_linear_zeros_bwd_ws_bytes": (_SZ, [_I, _I]),
    "lfi_linear_zeros_bwd": (_I, [_P, _P, _P, _P, _P, _F, _P, _P, _P, _P, _I, _I, _I, _P, _SZ, _P]),
    "lfi_fseq_ws_bytes": (_SZ, [_FS, _I]),
    "lfi_fseq_stash_bytes": (_SZ, [_FS, _I]),
    "lfi_fseq_bwd_ws_bytes": (_SZ, [_FS, _I]),
    "lfi_fseq_fwd": (_I, [_FS, _FP, _P, _P, _P, _P, _P, _P, _P, _I, _P, _SZ, _P, _SZ, _P]),
    "lfi_fseq_bwd": (_I, [_FS, _FP, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _FP, _I, _P, _SZ, _P, _SZ, _P]),
    "lfi_gather_batch": (_I, [_P, _P, _I, _I, _I, _P, _P]),
    "lfi_jerk": (_I, [_P, _I, _I, _I, _P, _P, _P]),
    "lfi_clip_adam": (_I, [_P, _P, _P, _P, _SZ, _F, _F, _F, _F, _F, _F, _I, _P, _P]),
    "lfi_clip_adam_dev": (_I, [_P, _P, _P, _P, _SZ, _P, _F, _F, _F, _F, _F, _P, _P]),
    "lfi_gemm": (_I, [_I, _I, _I, _I, _I, _I, _P, _I, _L, _P, _I, _L, _P, _I, _L, _P, _L, _P, _I, _L, _I, _I, _P, _SZ, _P]),
}

_lib = None


def lib():
    """Loads the shared library once; raises if it has not been built (no CPU / eager fallback)."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                "lets_face_it_b200: %s is missing - build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C lets_face_it_b200/csrc`); there is no fallback path." % LIB_PATH)
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(l, name)
            fn.restype, fn.argtypes = res, args
        if l.lfi_abi_version() != ABI_VERSION:
            raise RuntimeError("liblfi_b200.so ABI %d != binding ABI %d (stale build?)" % (l.lfi_abi_version(), ABI_VERSION))
        _lib = l
    return _lib


def check(status, what):
    if status != 0:
        msg = lib().lfi_last_error()
        raise RuntimeError("%s failed (status %d): %s" % (what, status, msg.decode() if msg else "?"))


def ptr(t):
    """Device pointer of a CUDA fp32 contiguous tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("lets_face_it_b200 kernels need CUDA tensors (got %s); there is no CPU path" % t.device)
    if t.dtype != _torch().float32 or not t.is_contiguous():
        raise RuntimeError("lets_face_it_b200 kernels need contiguous float32 tensors (got %s, contiguous=%s)" % (t.dtype, t.is_contiguous()))
    return t.data_ptr()


def _torch():
    import torch
    return torch


def stream_ptr():
    return _torch().cuda.current_stream().cuda_stream
