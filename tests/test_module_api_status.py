"""CPU: the module-API entry points of ABI 6 reject a missing or too-small workspace / stash with a status before they touch the
device (no compute: every call below returns from its argument checks)."""
import ctypes

from lets_face_it_b200 import _cabi

LFI_ERR_SHAPE, LFI_ERR_ARG, LFI_ERR_WORKSPACE = -1, -3, -4
FAKE = 1 << 20  # never dereferenced: the checks run first


def _shape(G=3):
    sh = _cabi.FseqShape()
    sh.In, sh.Out, sh.H, sh.D, sh.F, sh.G, sh.logscale_factor = 7, 3, 20, 24, 40, G, 3.0
    return sh


def _params():
    return _cabi.FseqParams(*([FAKE] * len(_cabi.FSEQ_PARAMS)))


def test_fseq_sizes():
    L = _cabi.lib()
    for G in (3, 4):
        sh = _shape(G)
        assert L.lfi_fseq_ws_bytes(ctypes.byref(sh), 21) > 0
        assert L.lfi_fseq_stash_bytes(ctypes.byref(sh), 21) > 0
        assert L.lfi_fseq_bwd_ws_bytes(ctypes.byref(sh), 21) > 0
    bad = _shape()
    bad.G = 5
    assert L.lfi_fseq_ws_bytes(ctypes.byref(bad), 21) == 0
    assert b"G=5" in L.lfi_last_error()
    assert L.lfi_fseq_stash_bytes(ctypes.byref(_shape()), 0) == 0
    assert L.lfi_linear_zeros_bwd_ws_bytes(21, 3) >= 21 * 3 * 4


def test_fseq_fwd_rejects_workspace_and_stash():
    L = _cabi.lib()
    sh, P, B = _shape(), _params(), 21
    ws = L.lfi_fseq_ws_bytes(ctypes.byref(sh), B)
    stash = L.lfi_fseq_stash_bytes(ctypes.byref(sh), B)
    args = lambda w, wb, s, sb: (ctypes.byref(sh), ctypes.byref(P), FAKE, FAKE, None, None, FAKE, None, FAKE, B, s, sb, w, wb, None)
    assert L.lfi_fseq_fwd(*args(None, ws, None, 0)) == LFI_ERR_ARG
    assert L.lfi_fseq_fwd(*args(FAKE, ws - 1, None, 0)) == LFI_ERR_WORKSPACE
    assert L.lfi_fseq_fwd(*args(FAKE, ws, FAKE, stash - 1)) == LFI_ERR_WORKSPACE
    lstm = _shape(4)
    assert L.lfi_fseq_fwd(ctypes.byref(lstm), ctypes.byref(P), FAKE, FAKE, None, None, FAKE, None, FAKE, B, None, 0, FAKE, 1 << 30,
                          None) == LFI_ERR_ARG  # LSTM without c_out
    assert L.lfi_fseq_fwd(*args(FAKE, ws, None, 0)[:9], 0, None, 0, FAKE, ws, None) == LFI_ERR_SHAPE


def test_fseq_bwd_rejects_workspace_and_stash():
    L = _cabi.lib()
    sh, P, G, B = _shape(), _params(), _params(), 21
    ws = L.lfi_fseq_bwd_ws_bytes(ctypes.byref(sh), B)
    stash = L.lfi_fseq_stash_bytes(ctypes.byref(sh), B)

    def call(w, wb, s, sb):
        return L.lfi_fseq_bwd(ctypes.byref(sh), ctypes.byref(P), FAKE, FAKE, None, None, FAKE, None, None, FAKE, FAKE, None, None,
                              ctypes.byref(G), B, s, sb, w, wb, None)

    assert call(None, ws, FAKE, stash) == LFI_ERR_ARG
    assert call(FAKE, ws, None, stash) == LFI_ERR_ARG
    assert call(FAKE, ws - 1, FAKE, stash) == LFI_ERR_WORKSPACE
    assert call(FAKE, ws, FAKE, stash - 1) == LFI_ERR_WORKSPACE


def test_linear_zeros_and_actnorm_bwd_reject_bad_arguments():
    L = _cabi.lib()
    B, In, Out = 21, 20, 7
    ws = L.lfi_linear_zeros_bwd_ws_bytes(B, Out)
    a = [FAKE] * 5
    assert L.lfi_linear_zeros_bwd(*a, 3.0, FAKE, FAKE, FAKE, FAKE, B, In, Out, None, ws, None) == LFI_ERR_ARG
    assert L.lfi_linear_zeros_bwd(*a, 3.0, FAKE, FAKE, FAKE, FAKE, B, In, Out, FAKE, ws - 1, None) == LFI_ERR_WORKSPACE
    assert L.lfi_actnorm_bwd(FAKE, None, FAKE, FAKE, FAKE, FAKE, FAKE, B, 13, 0, None) == LFI_ERR_ARG   # forward direction reads y
    assert L.lfi_actnorm_bwd(None, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, B, 13, 1, None) == LFI_ERR_ARG   # reverse reads x
    assert L.lfi_actnorm_bwd(FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, 0, 13, 0, None) == LFI_ERR_SHAPE
