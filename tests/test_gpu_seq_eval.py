"""GPU: SeqGlow.evaluate (lfi_seq_eval), the no-grad likelihood that scores a sequence in chunks of frames with the flow core's
RNN state carried from chunk to chunk.  Against the reference vectors, against the no-grad forward, across chunk sizes (where
the state carry is tested), on long sequences, and for its kernels, memory and lack of side effects."""
import copy
import ctypes

import pytest
import torch

from oracle import glow_oracle as O
from tests.helpers import final_hparams, golden_batch, golden_params, load_golden, relerr, small_hparams
from tests.kat import build_kat_model, kat_batch, to_device
from tests.test_gpu_core_plan import _core_path, _kernels

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
MODES = {"fp32": 0, "bf16x3": 1, "bf16": 2}
# bounds against the no-grad forward, as (z, nll) relative to the max: the encoders run other kernels (the persistent window
# GRU in the tensor-core modes, no stash), so the last bits differ
BOUNDS = {"fp32": (1e-5, 1e-5), "bf16x3": (1e-5, 1e-5), "bf16": (5e-3, 1e-4)}


def _final(mode, lstm_small=False, scale_logging=False):
    hp = copy.deepcopy(final_hparams())
    if lstm_small:
        hp.Glow.update(K=3, hidden_channels=64, rnn_type="lstm")
    hp.Validation["scale_logging"] = scale_logging
    m = build_kat_model(hp, DEV)
    m.glow.set_actnorm_init(True)
    m.gemm_mode = MODES[mode]
    m.eval()
    return m, hp


def _batch(hp, B, T, seed=5):
    return to_device(kat_batch(hp, B, T, seed=seed), DEV)


def _no_grad_forward(m, batch):
    with torch.no_grad():
        z, loss, losses = m(batch)
    return torch.stack(z), loss, torch.stack(losses)


def _evaluate(m, batch, chunk=None):
    z, loss, losses = m.evaluate(batch, chunk=chunk)
    return torch.stack(z), loss, torch.stack(losses)


# ------------------------------------------------------------------------------------------------ reference vectors
@pytest.mark.parametrize("rnn", ["gru", "lstm"])
@pytest.mark.parametrize("chunk", [None, 2])
def test_evaluate_matches_reference_vectors(rnn, chunk):
    from lets_face_it_b200.glow import ModalityEncoder, SeqGlow

    g = load_golden("kat_small_" + rnn)
    m = SeqGlow(small_hparams(rnn))
    m.load_state_dict(golden_params(g))
    for mod in m.modules():
        if isinstance(mod, ModalityEncoder):
            mod.dropout = None
    m.glow.set_actnorm_init(True)
    m = m.to(DEV).eval()
    batch = to_device(golden_batch(g), DEV)
    z_seq, loss, losses = m.evaluate(batch, chunk=chunk)
    assert len(z_seq) == g["z"].shape[0] and losses[0].device.type == "cpu" and loss.shape == (1,)
    assert not loss.requires_grad and not z_seq[0].requires_grad
    assert relerr(torch.stack(z_seq), g["z"]) < 1e-4
    assert relerr(torch.stack(losses), g["nll"]) < 1e-4
    assert abs(float(loss) - float(g["loss"][0])) < 1e-4 * abs(float(g["loss"][0]))


# ------------------------------------------------------------------------------------------------ against the no-grad forward
@pytest.mark.parametrize("mode", ["fp32", "bf16x3", "bf16"])
def test_evaluate_matches_no_grad_forward(mode):
    m, hp = _final(mode)
    batch = _batch(hp, 64, 80)
    z0, l0, n0 = _no_grad_forward(m, batch)
    z1, l1, n1 = _evaluate(m, batch)
    bz, bn = BOUNDS[mode]
    assert relerr(z1, z0) < bz
    assert relerr(n1, n0) < bn
    assert abs(float(l1) - float(l0)) < bn * abs(float(l0))


# ------------------------------------------------------------------------------------------------ chunk invariance (state carry)
@pytest.mark.parametrize("mode,tol", [("fp32", 1e-6), ("bf16x3", 1e-5)])
def test_chunks_agree_final_model(mode, tol):
    """40 scored frames.  The chunk changes the row count of the GEMMs, so their split-K choice and summation order."""
    m, hp = _final(mode)
    batch = _batch(hp, 64, 24 + 40)
    z, _, n = _evaluate(m, batch, chunk=40)
    for chunk in (1, 7, 64):
        zc, _, nc = _evaluate(m, batch, chunk=chunk)
        assert relerr(zc, z) < tol, chunk
        assert relerr(nc, n) < tol, chunk


def test_chunks_agree_small_lstm_wave():
    """LSTM, K = 3, H = 64: the wavefront kernels, with h and c carried between chunks."""
    m, hp = _final("fp32", lstm_small=True)
    batch = _batch(hp, 40, 24 + 13)
    z, _, n = _evaluate(m, batch, chunk=13)
    for chunk in (1, 4):
        zc, _, nc = _evaluate(m, batch, chunk=chunk)
        assert relerr(zc, z) < 1e-6, chunk
        assert relerr(nc, n) < 1e-6, chunk
    z0, _, n0 = _no_grad_forward(m, batch)
    assert relerr(z, z0) < 1e-5 and relerr(n, n0) < 1e-5


# ------------------------------------------------------------------------------------------------ long sequences
def test_prefix_of_a_long_sequence():
    m, hp = _final("bf16x3")
    batch = _batch(hp, 64, 24 + 600)
    z, _, n = _evaluate(m, batch)
    assert torch.isfinite(z).all() and torch.isfinite(n).all()
    zp, _, np_ = _evaluate(m, {k: v[:, :80].contiguous() for k, v in batch.items()})
    assert relerr(z[:56], zp) < 1e-5
    assert relerr(n[:56], np_) < 1e-5


# ------------------------------------------------------------------------------------------------ masks, FlowStep.scale
def test_injected_masks_in_training_mode():
    m, hp = _final("bf16x3")
    m.train()
    hy = O.Hyper.from_hparams(hp)
    masks = O.make_masks(hy, 64, 80 - hy.start_ts, seed=3)
    m.injected_masks = {k: (v.to(DEV) if v is not None else None) for k, v in masks.items()}
    assert any(v is not None for v in m.injected_masks.values())
    batch = _batch(hp, 64, 80)
    z0, _, n0 = _no_grad_forward(m, batch)
    z1, _, n1 = _evaluate(m, batch, chunk=5)
    assert relerr(z1, z0) < 1e-5
    assert relerr(n1, n0) < 1e-5


def test_flowstep_scale_under_scale_logging():
    m, hp = _final("bf16x3", scale_logging=True)
    batch = _batch(hp, 64, 80)
    _no_grad_forward(m, batch)
    s0 = [l.scale.clone() for l in m.glow.flow.layers]
    for l in m.glow.flow.layers:
        l.scale = None
    _evaluate(m, batch, chunk=7)
    s1 = [l.scale for l in m.glow.flow.layers]
    assert all(s is not None for s in s1)
    assert relerr(torch.stack(s1), torch.stack(s0)) < 1e-5


# ------------------------------------------------------------------------------------------------ kernels
@pytest.mark.parametrize("mode,env,lstm,core", [
    ("bf16x3", {}, False, "PipeTc"),
    ("bf16", {}, False, "PipeTc"),
    ("fp32", {}, False, "Pipe"),
    ("bf16x3", {"LFI_CORE_TC": "0"}, False, "Pipe"),
    ("bf16x3", {"LFI_CORE_PIPE": "0"}, False, "Wave"),
    ("bf16x3", {}, True, "Wave"),
])
def test_evaluate_kernels(mode, env, lstm, core, monkeypatch):
    """One chunk: the flow-core kernel of the plan (the carry instantiation of the pipelines), no backward kernel, and in
    bf16x3 at final shapes the persistent window-GRU encoder."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    m, hp = _final(mode, lstm_small=lstm)
    batch = _batch(hp, 64, 24 + 30)
    m.evaluate(batch, chunk=30)  # first call: workspace, function attributes
    names = _kernels(lambda: m.evaluate(batch, chunk=30))
    assert _core_path(names, "fwd") == core
    if core.startswith("Pipe"):
        fwd = [n for n in names if "core_fwd_pipe" in n]
        assert fwd and all("<true>" in n for n in fwd), fwd
    assert not any("bwd" in n for n in names), [n for n in names if "bwd" in n]
    if mode == "bf16x3" and not lstm and not env:
        assert any("enc_gru_fwd_persist" in n for n in names)


# ------------------------------------------------------------------------------------------------ memory
def test_long_sequence_memory():
    from lets_face_it_b200 import _cabi

    m, hp = _final("bf16x3")
    B, T = 256, 24 + 2000
    eng = m.engine()
    assert _cabi.lib().lfi_train_ws_bytes(ctypes.byref(eng.shape), B, T, _cabi.GEMM_BF16X3) > 400e9  # not run
    batch = _batch(hp, B, T)
    m.evaluate({k: v[:, :80].contiguous() for k, v in batch.items()})  # engine buffers, derived cache
    torch.cuda.synchronize()
    chunk = eng.eval_chunk(B, T)
    ws = _cabi.lib().lfi_eval_ws_bytes(ctypes.byref(eng.shape), B, T, chunk, _cabi.GEMM_BF16X3)
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    z, loss, losses = m.evaluate(batch)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    outputs = (T - 24) * B * (eng.C + 1) * 4
    assert len(z) == T - 24 and torch.isfinite(torch.stack(losses)).all()
    assert peak <= ws + outputs + (512 << 20), (peak, ws, outputs)


# ------------------------------------------------------------------------------------------------ no side effects
def test_no_side_effects_on_training():
    from lets_face_it_b200 import _cabi

    m, hp = _final("bf16x3")
    m.train()
    batch = _batch(hp, 64, 80)
    L = _cabi.lib()

    def step():
        m.zero_grad()
        n0 = L.lfi_launch_count()
        _, loss, _ = m(batch)
        loss.backward()
        torch.cuda.synchronize()
        g = torch.cat([p.grad.reshape(-1) for p in m.parameters() if p.grad is not None])
        return loss.detach().clone(), g.clone(), L.lfi_launch_count() - n0

    step()  # first call: workspaces
    l0, g0, c0 = step()
    m.evaluate(batch, chunk=7)
    l1, g1, c1 = step()
    assert torch.equal(l1, l0)
    assert c1 == c0
    # the backward pass sums some gradients with float atomics, so two steps agree to the last bits only up to their order
    assert relerr(g1, g0) < 1e-5
