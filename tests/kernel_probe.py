"""ctypes binding of the test-only probe library tests/_lib/liblfi_probe.so (source: tests/csrc/kernel_probe.cu).

The probe exports extern "C" wrappers around internal functions of liblfi_b200.so (the tcgen05 GEMM with its plane /
fused epilogues, the encoder aux kernels, the persistent window-GRU forward) and links against the shipped library, so
the tests drive the exact binary the package loads.  The argument structs below mirror csrc/lfi_common.cuh,
aux_kernels.cuh and enc_persist.cuh field by field; tests/test_kernel_probe_symbols.py compares them with the
compiler's layout (lfi_probe_layout).
"""
import ctypes as C
import os
import subprocess

from tests.helpers import ROOT

PROBE_SRC = os.path.join(ROOT, "tests", "csrc", "kernel_probe.cu")
PROBE_PATH = os.path.join(ROOT, "tests", "_lib", "liblfi_probe.so")
CSRC = os.path.join(ROOT, "lets_face_it_b200", "csrc")

FUSE_NONE, FUSE_GRU_FWD, FUSE_GRU_FWD_X = 0, 1, 3
EPI_ACCUM_PRE = 16

_P, _I, _L, _SZ = C.c_void_p, C.c_int, C.c_long, C.c_size_t


class PlaneRef(C.Structure):
    _fields_ = [("hi", _P), ("lo", _P), ("ld", _I), ("stride", _L)]


class GruEpi(C.Structure):
    _fields_ = [("E", _I), ("s", _I), ("hist", _I), ("B", _I), ("T", _I), ("t0", _I), ("gates16", _I),
                ("xp", _P), ("b_ih", _P), ("b_hh", _P), ("mask", _P), ("hprev", _P),
                ("h", _P), ("gates", _P), ("ahn", _P), ("cond", _P), ("cond_ld", _I),
                ("h_hi", _P), ("h_lo", _P),
                ("xa_hi", _P), ("xa_lo", _P), ("xb_hi", _P), ("xb_lo", _P), ("xa_ld", _I), ("xb_ld", _I), ("xk", _I),
                ("x_only", _I)]


class GemmArgs(C.Structure):
    _fields_ = [("transA", _I), ("transB", _I), ("M", _I), ("N", _I), ("K", _I),
                ("A", _P), ("lda", _I), ("sA", _L),
                ("B", _P), ("ldb", _I), ("sB", _L),
                ("C", _P), ("ldc", _I), ("sC", _L),
                ("bias", _P), ("sBias", _L),
                ("aux", _P), ("ldaux", _I), ("sAux", _L),
                ("batch", _I), ("epi", _I),
                ("pA", PlaneRef), ("pB", PlaneRef), ("pOut", PlaneRef),
                ("fuse", _I), ("gru", GruEpi),
                ("auxp", _P), ("ldauxp", _I), ("sAuxp", _L),
                ("colsum", _P), ("sColsum", _L),
                ("c_tiled32", _I)]


class EncStep(C.Structure):
    _fields_ = [("xp", _P), ("gh", _P), ("b_ih", _P), ("b_hh", _P), ("mask", _P), ("hprev", _P), ("h", _P),
                ("gates", _P), ("ahn", _P), ("cond", _P), ("cond_ld", _I), ("h_hi", _P), ("h_lo", _P),
                ("s", _I), ("hist", _I), ("B", _I), ("T", _I), ("Tp", _I), ("t0", _I), ("E", _I), ("gates16", _I)]


class EncStepBwd2(C.Structure):
    _fields_ = [("gates", _P), ("ahn", _P), ("hprev", _P), ("dh", _P), ("dh_extra", _P), ("dh_extra_ld", _I),
                ("dah32", _P), ("dan32", _P), ("dah_hi", _P), ("dah_lo", _P), ("dan_hi", _P), ("dan_lo", _P),
                ("gb_ih", _P), ("gb_hh", _P), ("M", _I), ("E", _I), ("gates16", _I)]


class FwdArgs(C.Structure):
    _fields_ = [("E", _I), ("hist", _I), ("B", _I), ("T", _I), ("t0", _I), ("M", _I), ("nplanes", _I),
                ("xp", _P), ("b_ih", _P), ("b_hh", _P), ("mask", _P), ("whh_hi", _P), ("whh_lo", _P),
                ("cond", _P), ("cond_ld", _I), ("timing", _I)]


STRUCTS = [PlaneRef, GruEpi, GemmArgs, EncStep, EncStepBwd2, FwdArgs]

SIGNATURES = {
    "lfi_probe_layout": (_SZ, [C.c_char_p, C.c_char_p]),
    "lfi_probe_gemm": (_I, [_I, C.POINTER(GemmArgs), _P, _SZ, _P]),
    "lfi_probe_gemm_ws_bytes": (_SZ, [_I, C.POINTER(GemmArgs)]),
    "lfi_probe_split_to_planes": (_I, [_P, _I, _I, _I, _L, _I, _P, _P, _P]),
    "lfi_probe_enc_gate_fwd": (_I, [C.POINTER(EncStep), _P]),
    "lfi_probe_enc_gate_bwd2": (_I, [C.POINTER(EncStepBwd2), _P]),
    "lfi_probe_colsum_planes": (_I, [_P, _P, _I, _I, _L, _P, _P, _I, _L, _I, _I, _I, _I, _P]),
    "lfi_probe_gather_windows_planes": (_I, [_P, _P, _I, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "lfi_probe_enc_fwd_supported": (_I, [_I, _I, _SZ, _I]),
    "lfi_probe_enc_launch_fwd": (_I, [C.POINTER(FwdArgs), _P]),
}

_lib = None


def _stale():
    if not os.path.isfile(PROBE_PATH):
        return True
    t = os.path.getmtime(PROBE_PATH)
    from lets_face_it_b200 import _cabi

    deps = [PROBE_SRC, _cabi.LIB_PATH] + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def lib():
    """Load the probe (building it with `make probe` when it is missing or older than its sources).  liblfi_b200.so is
    loaded first from the package, so the probe resolves its internal symbols against that same loaded image."""
    global _lib
    if _lib is not None:
        return _lib
    from lets_face_it_b200 import _cabi

    _cabi.lib()
    if _stale():
        r = subprocess.run(["make", "-C", CSRC, "probe"], capture_output=True, text=True)
        if r.returncode != 0 or not os.path.isfile(PROBE_PATH):
            raise RuntimeError("could not build the kernel probe %s with `make -C %s probe`:\n%s\n%s"
                               % (PROBE_PATH, CSRC, r.stdout[-2000:], r.stderr[-4000:]))
    l = C.CDLL(PROBE_PATH)
    for name, (res, args) in SIGNATURES.items():
        f = getattr(l, name)
        f.restype = res
        f.argtypes = args
    _lib = l
    return l


def layout(type_name, field=""):
    return int(lib().lfi_probe_layout(type_name.encode(), field.encode()))


def check(status, what):
    from lets_face_it_b200 import _cabi

    _cabi.check(status, what)
