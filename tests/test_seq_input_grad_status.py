"""CPU: the input-gradient backward of ABI 8 (lfi_seq_train_bwd_dx) sizes its dXg scratch (lfi_train_dx_ws_bytes) and rejects null
pointers, a gradient asked for an absent modality and short workspaces with a status before it launches anything (no compute:
every call below returns from its argument checks, and the library's launch counter does not move)."""
import ctypes

from lets_face_it_b200 import _cabi
from lets_face_it_b200.engine import MODALITIES
from lets_face_it_b200.hparams import load_hparams

LFI_ERR_SHAPE, LFI_ERR_ARG, LFI_ERR_WORKSPACE = -1, -3, -4
FAKE = 1 << 20  # never dereferenced: the checks run first
B, T = 256, 80


def _final_shape():
    """final_model.yaml: p1_face enc: none (hist 5), p2_face GRU (24, 56, 256), p1_speech GRU (2, 30, 128), p2_speech GRU (16, 30, 256)."""
    hp = load_hparams()
    sh = _cabi.Shape()
    sh.C, sh.K, sh.H, sh.D, sh.G, sh.affine, sh.scale_eps, sh.f_raw = 56, 16, 128, 512, 3, 1, 1e-4, 0
    for i, m in enumerate(MODALITIES):
        c = hp.Conditioning[m]
        sh.hist[i] = c["history"]
        sh.dim[i] = c.get("dim", hp.Data["speech_dim"])
        sh.ehid[i] = c["hidden_dim"] if c["enc"] == "rnn" else 0
    return sh


def test_dx_ws_bytes_final_model():
    L = _cabi.lib()
    sh = _final_shape()
    start = L.lfi_start_ts(ctypes.byref(sh))
    assert start == 24
    M = (T - start) * B
    # one fp32 dXg [hist * M, dim] per GRU modality, 256-byte aligned
    want = sum(-(-sh.hist[i] * M * sh.dim[i] * 4 // 256) * 256 for i in range(_cabi.NMOD) if sh.hist[i] > 0 and sh.ehid[i] > 0)
    assert want == 108_036_096
    for mode in (_cabi.GEMM_FP32, _cabi.GEMM_BF16X3, _cabi.GEMM_BF16):
        assert L.lfi_train_dx_ws_bytes(ctypes.byref(sh), B, T, mode) == want
    # more frames, more scratch
    assert L.lfi_train_dx_ws_bytes(ctypes.byref(sh), B, T + 1, 1) > want


def test_dx_ws_bytes_without_encoders_and_bad_shapes():
    L = _cabi.lib()
    sh = _final_shape()
    for i in range(_cabi.NMOD):
        sh.ehid[i] = 0  # every modality "enc: none": no dXg scratch, only the minimal allocation
    assert L.lfi_train_dx_ws_bytes(ctypes.byref(sh), B, T, 1) == 256
    sh.hist[1] = sh.hist[2] = sh.hist[3] = 0
    assert L.lfi_train_dx_ws_bytes(ctypes.byref(sh), B, T, 1) == 256
    good = _final_shape()
    assert L.lfi_train_dx_ws_bytes(ctypes.byref(good), 0, T, 1) == 0   # B < 1
    assert L.lfi_train_dx_ws_bytes(ctypes.byref(good), B, 24, 1) == 0  # no trained frame
    bad = _final_shape()
    bad.G = 5
    assert L.lfi_train_dx_ws_bytes(ctypes.byref(bad), B, T, 1) == 0
    assert b"G=5" in L.lfi_last_error()


def _params():
    P = _cabi.Params()
    for f in ("an_bias", "an_logs", "w", "wc", "bc", "w_ih", "b_ih", "w_hh", "b_hh", "wf", "bf", "lf"):
        setattr(P, f, FAKE)
    for name in ("enc_w_ih", "enc_w_hh", "enc_b_ih", "enc_b_hh"):
        for i in range(1, _cabi.NMOD):
            getattr(P, name)[i] = FAKE
    return P


def _batch(sh):
    bt = _cabi.Batch()
    bt.B, bt.T = B, T
    for i in range(_cabi.NMOD):
        bt.x[i] = FAKE if sh.hist[i] > 0 else None
    return bt


def test_bwd_dx_rejects_arguments_before_launching():
    L = _cabi.lib()
    sh = _final_shape()
    P, G, bt = _params(), _params(), _batch(sh)
    ws = L.lfi_train_ws_bytes(ctypes.byref(sh), B, T, 1)
    dws = L.lfi_train_dx_ws_bytes(ctypes.byref(sh), B, T, 1)
    every = (ctypes.c_void_p * _cabi.NMOD)(FAKE, FAKE, FAKE, FAKE)

    def call(dx=every, derived=FAKE, z=FAKE, dnll=FAKE, grads=G, w=FAKE, wb=ws, d=FAKE, db=dws, shape=sh):
        return L.lfi_seq_train_bwd_dx(ctypes.byref(shape), derived, ctypes.byref(P), ctypes.byref(bt), z, dnll, ctypes.byref(grads), w, wb,
                                      dx, d, db, 1, None)

    n0 = L.lfi_launch_count()
    assert call(dx=None) == LFI_ERR_ARG
    assert call(derived=None) == LFI_ERR_ARG
    assert call(z=None) == LFI_ERR_ARG
    assert call(dnll=None) == LFI_ERR_ARG
    assert call(w=None) == LFI_ERR_ARG
    assert call(d=None) == LFI_ERR_ARG
    assert b"dx workspace" in L.lfi_last_error()
    assert call(wb=ws - 1) == LFI_ERR_WORKSPACE
    assert call(db=dws - 1) == LFI_ERR_WORKSPACE
    assert b"dx workspace too small" in L.lfi_last_error()
    # a gradient asked for a modality the shape does not have
    part = _final_shape()
    part.hist[3] = 0
    pws = L.lfi_train_ws_bytes(ctypes.byref(part), B, T, 1)
    pdws = L.lfi_train_dx_ws_bytes(ctypes.byref(part), B, T, 1)
    assert call(shape=part, wb=pws, db=pdws) == LFI_ERR_ARG
    assert b"absent modality" in L.lfi_last_error()
    assert L.lfi_launch_count() == n0
