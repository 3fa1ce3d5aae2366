"""CPU: the encoder entry points of ABI 7 (lfi_feature_encode_fwd_train / lfi_feature_encode_bwd) size their stash and workspace,
reject a bad shape with an error text, and reject a missing or too-small stash / workspace with a status before they touch the
device (no compute: every call below returns from its argument checks)."""
import ctypes

from lets_face_it_b200 import _cabi

LFI_ERR_SHAPE, LFI_ERR_ARG, LFI_ERR_WORKSPACE = -1, -3, -4
FAKE = 1 << 20  # never dereferenced: the checks run first
B, T, TP = 16, 30, 3


def _shape():
    """final_model.yaml's encoders (p1_face enc: none, three GRUs) with a small flow."""
    sh = _cabi.Shape()
    sh.C, sh.K, sh.H, sh.D, sh.G, sh.affine, sh.scale_eps, sh.f_raw = 56, 2, 16, 24, 3, 1, 1e-4, 0
    for i, (h, d, e) in enumerate([(5, 56, 0), (24, 56, 256), (2, 30, 128), (16, 30, 256)]):
        sh.hist[i], sh.dim[i], sh.ehid[i] = h, d, e
    return sh


def _params():
    P = _cabi.Params()
    for name in ("enc_w_ih", "enc_w_hh", "enc_b_ih", "enc_b_hh"):
        for i in range(1, _cabi.NMOD):
            getattr(P, name)[i] = FAKE
    return P


def _batch():
    bt = _cabi.Batch()
    bt.B, bt.T = B, T
    for i in range(_cabi.NMOD):
        bt.x[i] = FAKE
    return bt


def test_sizes():
    L = _cabi.lib()
    sh = _shape()
    for mode in (_cabi.GEMM_FP32, _cabi.GEMM_BF16X3, _cabi.GEMM_BF16):
        assert L.lfi_feature_stash_bytes(ctypes.byref(sh), B, T, TP, mode) > 0
        assert L.lfi_feature_bwd_ws_bytes(ctypes.byref(sh), B, T, TP, mode) > 0
    # more windows per call, a larger stash
    assert L.lfi_feature_stash_bytes(ctypes.byref(sh), B, T, TP + 1, 0) > L.lfi_feature_stash_bytes(ctypes.byref(sh), B, T, TP, 0)
    bad = _shape()
    bad.G = 5
    assert L.lfi_feature_stash_bytes(ctypes.byref(bad), B, T, TP, 0) == 0
    assert b"G=5" in L.lfi_last_error()
    assert L.lfi_feature_bwd_ws_bytes(ctypes.byref(bad), B, T, TP, 0) == 0
    raw = _shape()
    raw.f_raw = 40
    assert L.lfi_feature_stash_bytes(ctypes.byref(raw), B, T, TP, 0) == 0
    assert b"f_raw" in L.lfi_last_error()
    assert L.lfi_feature_stash_bytes(ctypes.byref(sh), 0, T, TP, 0) == 0
    assert L.lfi_feature_bwd_ws_bytes(ctypes.byref(sh), B, T, 0, 0) == 0
    assert L.lfi_feature_bwd_ws_bytes(ctypes.byref(sh), B, T, TP, 7) == 0


def test_fwd_train_rejects_arguments():
    L = _cabi.lib()
    sh, P, bt = _shape(), _params(), _batch()
    stash = L.lfi_feature_stash_bytes(ctypes.byref(sh), B, T, TP, 0)
    ws = L.lfi_feature_bwd_ws_bytes(ctypes.byref(sh), B, T, TP, 0)
    t0 = L.lfi_start_ts(ctypes.byref(sh))

    def call(s, sb, w, wb, t=t0, params=P):
        return L.lfi_feature_encode_fwd_train(ctypes.byref(sh), ctypes.byref(params), ctypes.byref(bt), t, TP, FAKE, s, sb, w, wb, 0, None)

    assert call(None, stash, FAKE, ws) == LFI_ERR_ARG
    assert call(FAKE, stash, None, ws) == LFI_ERR_ARG
    assert call(FAKE, stash - 1, FAKE, ws) == LFI_ERR_WORKSPACE
    assert call(FAKE, stash, FAKE, ws - 1) == LFI_ERR_WORKSPACE
    assert call(FAKE, stash, FAKE, ws, t=t0 - 1) == LFI_ERR_SHAPE      # window would start before frame 0
    assert call(FAKE, stash, FAKE, ws, t=T - TP + 1) == LFI_ERR_SHAPE  # frames past the batch
    assert call(FAKE, stash, FAKE, ws, params=_cabi.Params()) == LFI_ERR_ARG  # GRU weights missing
    assert b"weights missing" in L.lfi_last_error()


def test_bwd_rejects_arguments():
    L = _cabi.lib()
    sh, P, G, bt = _shape(), _params(), _params(), _batch()
    stash = L.lfi_feature_stash_bytes(ctypes.byref(sh), B, T, TP, 1)
    ws = L.lfi_feature_bwd_ws_bytes(ctypes.byref(sh), B, T, TP, 1)
    t0 = L.lfi_start_ts(ctypes.byref(sh))
    dx = (ctypes.c_void_p * _cabi.NMOD)(FAKE, None, FAKE, None)

    def call(s, sb, w, wb, grads=G, dcond=FAKE):
        return L.lfi_feature_encode_bwd(ctypes.byref(sh), ctypes.byref(P), ctypes.byref(bt), t0, TP, dcond, dx, ctypes.byref(grads), s, sb, w, wb,
                                        1, None)

    assert call(None, stash, FAKE, ws) == LFI_ERR_ARG
    assert call(FAKE, stash, None, ws) == LFI_ERR_ARG
    assert call(FAKE, stash, FAKE, ws, dcond=None) == LFI_ERR_ARG
    assert call(FAKE, stash - 1, FAKE, ws) == LFI_ERR_WORKSPACE
    assert call(FAKE, stash, FAKE, ws - 1) == LFI_ERR_WORKSPACE
    assert call(FAKE, stash, FAKE, ws, grads=_cabi.Params()) == LFI_ERR_ARG  # gradient pointers missing
    assert b"gradients missing" in L.lfi_last_error()
