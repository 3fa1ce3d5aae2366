"""GPU test of which flow-core kernels one training step runs (core_plan.cu: plan_core): the profiler lists the kernels of the
forward and of the backward call, for final_model.yaml shapes in each GEMM mode, under each switch of DESIGN.md §9 that
selects a flow-core path, and for a small LSTM shape outside the stage pipelines."""
import copy

import pytest
import torch

from tests.helpers import final_hparams
from tests.kat import build_kat_model, kat_batch, to_device

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CORE = ("core_fwd_pipe_tc", "core_fwd_pipe", "core_fwd_wave", "core_bwd_pipe_tc", "core_bwd_pipe", "core_bwd_wave")


def _kernels(fn):
    """Names of the kernels fn launches, in the order they started on the device."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if e.device_type == DeviceType.CUDA and not e.name.startswith(("Memcpy", "Memset"))]
    return [e.name for e in sorted(ev, key=lambda e: e.time_range.start)]


def _core_path(names, direction):
    """'PipeTc', 'Pipe', 'WaveHybrid' or 'Wave': the flow-core kernel of one direction.  Hybrid wavefronts issue a batched
    recurrent GEMM between consecutive wavefront launches; the plain ones launch the wavefronts back to back."""
    cores = [next((c for c in CORE if c in n), None) for n in names]  # (CORE lists "_pipe_tc" first)
    found = {c for c in cores if c and c.startswith("core_" + direction)}
    assert len(found) == 1, (direction, found)
    kind = found.pop()
    if kind.endswith("_pipe_tc"):
        return "PipeTc"
    if kind.endswith("_pipe"):
        return "Pipe"
    idx = [i for i, c in enumerate(cores) if c == kind]
    between = cores[idx[0]:idx[-1]].count(None)
    if between == 0:
        return "Wave"
    assert between >= len(idx) - 1, (direction, between, len(idx))
    return "WaveHybrid"


def _step(hp, mode, B, T):
    from lets_face_it_b200 import _cabi as cabi

    m = build_kat_model(hp, DEV)
    m.glow.set_actnorm_init(True)
    m.gemm_mode = {"fp32": cabi.GEMM_FP32, "bf16x3": cabi.GEMM_BF16X3, "bf16": cabi.GEMM_BF16}[mode]
    m.train()
    batch = to_device(kat_batch(hp, B, T, seed=5), DEV)
    out = {}

    def fwd():
        out["loss"] = m(batch)[1]

    fwd()  # first call: workspaces, derived cache, function attributes
    out["loss"].backward()
    m.zero_grad()
    f = _kernels(fwd)
    b = _kernels(lambda: out["loss"].backward())
    return _core_path(f, "fwd"), _core_path(b, "bwd")


@pytest.mark.parametrize("mode,env,fwd,bwd", [
    ("fp32", {}, "Pipe", "Pipe"),
    ("bf16x3", {}, "PipeTc", "PipeTc"),
    ("bf16", {}, "PipeTc", "PipeTc"),
    ("bf16x3", {"LFI_CORE_TC": "0"}, "Pipe", "Pipe"),
    ("bf16x3", {"LFI_CORE_TC_BWD": "0"}, "PipeTc", "Pipe"),
    ("bf16x3", {"LFI_CORE_PIPE": "0"}, "WaveHybrid", "WaveHybrid"),
    ("bf16x3", {"LFI_WAVE_TC": "0"}, "PipeTc", "PipeTc"),
    ("fp32", {"LFI_CORE_PIPE": "0"}, "Wave", "Wave"),
])
def test_final_model_core_kernels(mode, env, fwd, bwd, monkeypatch):
    """final_model.yaml (GRU, H = 128, K = 16), B = 64, three trained frames."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    hp = final_hparams()
    assert _step(hp, mode, 64, 27) == (fwd, bwd)


@pytest.mark.parametrize("mode,env,fwd,bwd", [
    ("bf16x3", {}, "WaveHybrid", "WaveHybrid"),
    ("bf16x3", {"LFI_WAVE_TC": "0"}, "Wave", "Wave"),
    ("fp32", {}, "Wave", "Wave"),
])
def test_small_lstm_core_kernels(mode, env, fwd, bwd, monkeypatch):
    """LSTM, H = 64, K = 3 (no stage pipeline), B = 40, six trained frames."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    hp = copy.deepcopy(final_hparams())
    hp.Glow.update(K=3, hidden_channels=64, rnn_type="lstm")
    assert _step(hp, mode, 40, 30) == (fwd, bwd)
