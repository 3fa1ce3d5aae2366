"""CPU (no device): workspace sizes of the time-chunked likelihood evaluation (lfi_eval_ws_bytes) and the argument checks of
lfi_seq_eval / SeqGlow.evaluate, which return or raise before anything is launched."""
import ctypes

import pytest
import torch

from lets_face_it_b200 import _cabi
from lets_face_it_b200.engine import MODALITIES
from tests.helpers import final_hparams, small_hparams

MODES = (_cabi.GEMM_FP32, _cabi.GEMM_BF16X3, _cabi.GEMM_BF16)


def _final_shape():
    hp = final_hparams()
    sh = _cabi.Shape()
    sh.C, sh.K, sh.H, sh.D, sh.G, sh.affine, sh.scale_eps = 56, 16, 128, 512, 3, 1, 1e-4
    for i, m in enumerate(MODALITIES):
        c = hp.Conditioning[m]
        sh.hist[i] = c["history"]
        sh.dim[i] = c.get("dim", hp.Data["speech_dim"])
        sh.ehid[i] = c["hidden_dim"] if c["enc"] == "rnn" else 0
    return sh


def _eval_bytes(sh, B, T, chunk, mode):
    return _cabi.lib().lfi_eval_ws_bytes(ctypes.byref(sh), B, T, chunk, mode)


def test_eval_ws_bytes_bad_arguments():
    sh = _final_shape()
    assert _eval_bytes(sh, 64, 80, 8, _cabi.GEMM_BF16X3) > 0
    assert _eval_bytes(sh, 64, 80, 0, _cabi.GEMM_BF16X3) == 0    # chunk < 1
    assert _eval_bytes(sh, 64, 24, 8, _cabi.GEMM_BF16X3) == 0    # T <= start_ts
    assert _eval_bytes(sh, 0, 80, 8, _cabi.GEMM_BF16X3) == 0     # B < 1
    bad = _final_shape()
    bad.H = 130                                                  # H not a multiple of 4
    assert _eval_bytes(bad, 64, 80, 8, _cabi.GEMM_BF16X3) == 0


@pytest.mark.parametrize("mode", MODES)
def test_eval_ws_below_a_third_of_training(mode):
    sh = _final_shape()
    train = _cabi.lib().lfi_train_ws_bytes(ctypes.byref(sh), 256, 80, mode)
    assert 0 < _eval_bytes(sh, 256, 80, 56, mode) < train / 3


@pytest.mark.parametrize("mode", MODES)
def test_eval_ws_grows_only_by_the_encoder_projections(mode):
    """From T to T + 1,000 frames the workspace grows by no more than the encoders' per-raw-frame input projections (4 * 3E bytes
    per GRU modality) and, on the persistent encoder path (tensor-core modes), the time-major raw frames in fp32 and as the
    projection GEMM's bf16 operand planes."""
    sh = _final_shape()
    B, T, dT = 256, 80, 1000
    grow = _eval_bytes(sh, B, T + dT, 56, mode) - _eval_bytes(sh, B, T, 56, mode)
    gru = [i for i in range(_cabi.NMOD) if sh.hist[i] > 0 and sh.ehid[i] > 0]
    per_frame = sum(4 * 3 * sh.ehid[i] for i in gru)
    if mode != _cabi.GEMM_FP32:
        planes = 2 if mode == _cabi.GEMM_BF16X3 else 1
        per_frame += sum(4 * sh.dim[i] for i in gru) + 2 * planes * max(sh.dim[i] for i in range(_cabi.NMOD) if sh.hist[i] > 0)
    assert 0 < grow <= B * dT * per_frame + (1 << 20), (grow, B * dT * per_frame)


@pytest.mark.parametrize("mode", MODES)
def test_eval_ws_of_a_long_sequence(mode):
    sh = _final_shape()
    assert 0 < _eval_bytes(sh, 256, 24 + 10000, 56, mode) < 32e9


def _call(sh, derived=1, params=True, batch=True, chunk=4, z=1, nll=1, ws=1, ws_bytes=1 << 40, B=64, T=80):
    L = _cabi.lib()
    P = _cabi.Params()
    bt = _cabi.Batch()
    bt.B, bt.T = B, T
    bt.x[0] = 1
    return L.lfi_seq_eval(ctypes.byref(sh), derived, ctypes.byref(P) if params else None, ctypes.byref(bt) if batch else None,
                          chunk, z, nll, None, ws, ws_bytes, _cabi.GEMM_BF16X3, None)


def test_seq_eval_rejects_bad_arguments_before_launching():
    """Non-null dummies stand in for device pointers: every call fails its checks before touching them."""
    sh = _final_shape()
    ERR_ARG, ERR_WS = -3, -4
    assert _call(sh, derived=None) == ERR_ARG
    assert _call(sh, params=False) == ERR_ARG
    assert _call(sh, batch=False) == ERR_ARG
    assert _call(sh, z=None) == ERR_ARG
    assert _call(sh, nll=None) == ERR_ARG
    assert _call(sh, ws=None) == ERR_ARG
    assert _call(sh, chunk=0) == ERR_ARG
    assert _call(sh, T=24) == ERR_ARG                                  # T <= start_ts
    need = _eval_bytes(sh, 64, 80, 4, _cabi.GEMM_BF16X3)
    assert _call(sh, ws_bytes=need - 1) == ERR_WS
    assert b"eval workspace too small" in _cabi.lib().lfi_last_error()


def test_evaluate_on_cpu_tensors_raises():
    from lets_face_it_b200.glow import SeqGlow

    m = SeqGlow(small_hparams())
    batch = {"p1_face": torch.zeros(2, 12, 12), "p2_face": torch.zeros(2, 12, 12), "p1_speech": torch.zeros(2, 12, 5),
             "p2_speech": torch.zeros(2, 12, 5)}
    with pytest.raises(RuntimeError):
        m.evaluate(batch)
