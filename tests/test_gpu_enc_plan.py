"""GPU test of which window-GRU encoder kernels run (seq.cu: plan_enc): the profiler lists the kernels of one training forward,
one feature encoding and one short autoregressive sampling call.  final_model.yaml shapes (p2_face, p1_speech, p2_speech at
E = 256 / 128 / 256, hist = 24 / 2 / 16: 42 window steps) in each GEMM mode, under each switch of DESIGN.md §9 that selects an
encoder path, and with p2_speech at E = 96 (no fused step) or E = 24 (below the operand-plane minimum of 32)."""
import copy
import re
from collections import Counter

import pytest

from tests.helpers import final_hparams
from tests.kat import build_kat_model, kat_batch, to_device
from tests.test_gpu_core_plan import _kernels

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
B, T = 64, 27  # start_ts = 24: three frames, M = 192 windows
STEP_KINDS = ("fusedx", "fused", "gate", "persist")


def _kind(name):
    m = re.search(r"gemm_tc_kernel<(\d+),", name)
    if m:
        return {"0": "gemm", "1": "fused", "3": "fusedx"}[m.group(1)]  # LFI_FUSE_NONE, _GRU_FWD, _GRU_FWD_X
    for part, kind in (("gemm_simt_kernel", "gemm_simt"), ("split_planes_kernel", "split"), ("enc_gate_fwd", "gate"),
                       ("enc_gru_fwd_persist", "persist")):
        if part in name:
            return kind
    return None


def _encoder_kernels(names):
    """Window-step kernels of each kind; the tcgen05 GEMMs before the first window step (the encoders' input projections:
    nothing else ahead of the recurrences runs on those tiles); the GEMMs and operand splits between the first and the last
    window step (the recurrent products of the unfused steps)."""
    kinds = [_kind(n) for n in names]
    steps = [i for i, k in enumerate(kinds) if k in STEP_KINDS]
    first, last = steps[0], steps[-1]
    count = Counter(kinds)
    out = {k: count[k] for k in STEP_KINDS}
    out["proj"] = kinds[:first].count("gemm")
    for k in ("gemm", "gemm_simt", "split"):
        out["rec_" + k] = kinds[first:last].count(k)
    return out


def _model(mode, p2_speech_E=None):
    from lets_face_it_b200 import _cabi as cabi

    hp = final_hparams()
    if p2_speech_E is not None:
        hp = copy.deepcopy(hp)
        hp.Conditioning["p2_speech"]["hidden_dim"] = p2_speech_E
    m = build_kat_model(hp, DEV)
    m.glow.set_actnorm_init(True)
    m.gemm_mode = {"fp32": cabi.GEMM_FP32, "bf16x3": cabi.GEMM_BF16X3, "bf16": cabi.GEMM_BF16}[mode]
    return hp, m, to_device(kat_batch(hp, B, T, seed=5), DEV)


def _profiled(fn):
    fn()  # first call: workspaces, derived cache, function attributes
    return _encoder_kernels(_kernels(fn))


def _training_forward(mode, p2_speech_E=None):
    _, m, batch = _model(mode, p2_speech_E)
    m.train()
    return _profiled(lambda: m(batch))


def _subset(got, expect):
    return {k: got[k] for k in expect}


@pytest.mark.parametrize("mode,env,expect", [
    ("bf16x3", {}, dict(fusedx=42, fused=0, gate=0, persist=0, proj=0)),
    ("bf16", {}, dict(fusedx=42, fused=0, gate=0, persist=0, proj=0)),
    ("bf16x3", {"LFI_ENC_XFUSE": "0"}, dict(fusedx=0, fused=39, gate=3, persist=0, proj=3)),
    ("fp32", {}, dict(fusedx=0, fused=0, gate=42, persist=0, rec_gemm_simt=39)),
])
def test_training_forward_encoder_kernels(mode, env, expect, monkeypatch):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    assert _subset(_training_forward(mode), expect) == expect


@pytest.mark.parametrize("call", ["feature_encode", "inference"])
@pytest.mark.parametrize("env,expect", [
    ({}, dict(fusedx=0, fused=0, gate=0, persist=3, proj=3)),
    ({"LFI_ENC_PERSIST_SAMPLE": "0"}, dict(fusedx=0, fused=39, gate=3, persist=0, proj=3)),
])
def test_feature_encoding_and_sampling_encoder_kernels(call, env, expect, monkeypatch):
    """bf16x3.  Feature encoding of the three frames; sampling of three frames after the 24 seed frames (one chunk)."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    _, m, batch = _model("bf16x3")
    m.eval()
    if call == "feature_encode":
        eng = m.engine()
        got = _profiled(lambda: eng.feature_encode(batch, eng.start_ts, T - eng.start_ts))
    else:
        got = _profiled(lambda: m.inference(T, data=batch))
    assert _subset(got, expect) == expect


@pytest.mark.parametrize("E,expect", [
    # on operand planes: the recurrent GEMMs read the h and W_hh planes, nothing is split per step
    (96, dict(fusedx=26, fused=0, gate=16, proj=1, rec_gemm=15, rec_gemm_simt=0, rec_split=0)),
    # fp32 operands: [192, 24] x [24, 72] is too small for the tcgen05 tiles
    (24, dict(fusedx=26, fused=0, gate=16, proj=1, rec_gemm=0, rec_gemm_simt=15, rec_split=0)),
])
def test_unfused_encoder_kernels(E, expect):
    """bf16x3 training forward with p2_speech (16 window steps) at E % 64 != 0: its steps are a recurrent GEMM and a gate
    kernel each, after p2_face and p1_speech on the fused steps (the chains run one after another)."""
    assert _subset(_training_forward("bf16x3", E), expect) == expect
