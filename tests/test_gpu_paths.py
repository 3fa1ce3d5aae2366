"""GPU tests of the fast paths at BASELINE.json sizes: the stage-pipelined flow core against the general wavefront
kernels, the tensor-core sampler against the in-kernel fp32 sampler, and size-independent properties (forward ->
invert round trip, batch-shard equivalence) in the tensor-core modes the bench runs in.  Everything goes through the
module API -> C ABI; the oracle is only the checker."""
import os

import pytest
import torch

from oracle import glow_oracle as O
from tests.helpers import final_hparams, relerr
from tests.kat import build_kat_model, kat_batch, oracle_params_from, to_device

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


class _env:
    """Environment switches of the library are read at call time (getenv inside the C ABI)."""

    def __init__(self, **kv):
        self.kv, self.old = kv, {}

    def __enter__(self):
        for k, v in self.kv.items():
            self.old[k] = os.environ.get(k)
            os.environ[k] = v

    def __exit__(self, *a):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _model(mode):
    from lets_face_it_b200 import _cabi as cabi

    hp = final_hparams()
    m = build_kat_model(hp, DEV)
    m.glow.set_actnorm_init(True)
    m.gemm_mode = {"fp32": cabi.GEMM_FP32, "bf16x3": cabi.GEMM_BF16X3, "bf16": cabi.GEMM_BF16}[mode]
    return hp, m


def _fwd_bwd(m, batch):
    m.zero_grad()
    z_seq, loss, losses = m(batch)
    loss.backward()
    g = {n: p.grad.detach().clone() for n, p in m.named_parameters()}
    return torch.stack(z_seq).detach().clone(), torch.stack(losses).detach().clone(), g


@pytest.mark.parametrize("B", [256, 100])
def test_pipelined_core_matches_wavefront_kernels(B):
    """final_model.yaml, T=80: the persistent stage-pipelined core (2-CTA clusters, weights resident in shared memory) and
    the general wavefront kernels are two schedules of the same arithmetic: z / NLL to 1e-5, gradients to 1e-4 (fp32
    summation order differs).  B=100 leaves a ragged second tile (36 rows: the second CTA of the cluster owns 4)."""
    hp, m = _model("fp32")
    m.train()
    batch = to_device(kat_batch(hp, B, 80, seed=11), DEV)
    z1, n1, g1 = _fwd_bwd(m, batch)
    with _env(LFI_CORE_PIPE="0"):
        z0, n0, g0 = _fwd_bwd(m, batch)
    assert relerr(z1, z0) < 1e-5
    assert relerr(n1, n0) < 1e-5
    for k in g0:
        ref = g0[k].double()
        err = float((g1[k].double() - ref).norm() / ref.norm().clamp_min(1e-30))
        assert err < 1e-4, (k, err)


@pytest.mark.parametrize("B", [256, 100])
def test_tensor_core_flow_core_matches_ffma_core(B):
    """Tensor-core modes, final_model.yaml, T=80: the forward flow core with its recurrent / z1 / LinearZeros products as
    tcgen05.mma on split-bf16 operand planes (tiled gate stash, read by the backward pipeline) against the FFMA pipeline
    (LFI_CORE_TC=0, row-major stash) in the same GEMM mode: z / NLL within 5e-5 (three-product split-bf16 is fp32-grade),
    per-tensor gradients within 2e-3 relative L2; and z within the 1e-4 parity gate of the fp32 wavefront kernels.
    B=100 leaves a ragged second tile whose padding rows live only in the tiled stash."""
    hp, m = _model("bf16x3")
    m.train()
    batch = to_device(kat_batch(hp, B, 80, seed=14), DEV)
    z1, n1, g1 = _fwd_bwd(m, batch)
    with _env(LFI_CORE_TC="0"):
        z0, n0, g0 = _fwd_bwd(m, batch)
    assert relerr(z1, z0) < 5e-5
    assert relerr(n1, n0) < 5e-5
    for k in g0:
        ref = g0[k].double()
        err = float((g1[k].double() - ref).norm() / ref.norm().clamp_min(1e-30))
        assert err < 2e-3, (k, err)
    from lets_face_it_b200 import _cabi as cabi

    m.gemm_mode = cabi.GEMM_FP32
    with _env(LFI_CORE_PIPE="0"):
        z32, n32, _ = _fwd_bwd(m, batch)
    assert relerr(z1, z32) < 1e-4
    assert relerr(n1, n32) < 1e-4


def test_bf16_backward_option_stays_inside_gradient_bound():
    """LFI_BWD_BF16=1 (an option bench.py reports next to the headline): forward unchanged bit for bit, time-parallel backward
    GEMMs with single bf16 products - per-tensor gradients within the stated 5e-3 relative L2 of the split-bf16 backward."""
    hp, m = _model("bf16x3")
    m.train()
    batch = to_device(kat_batch(hp, 256, 80, seed=15), DEV)
    z0, n0, g0 = _fwd_bwd(m, batch)
    with _env(LFI_BWD_BF16="1"):
        z1, n1, g1 = _fwd_bwd(m, batch)
    assert torch.equal(z0, z1) and torch.equal(n0, n1)
    for k in g0:
        ref = g0[k].double()
        err = float((g1[k].double() - ref).norm() / ref.norm().clamp_min(1e-30))
        assert err < 5e-3, (k, err)


def test_full_size_roundtrip_and_sharding_in_parity_mode():
    """BASELINE configs[1] size (B=256, T=80) in the bf16x3 mode the bench runs in: forward -> invert reproduces the input
    frames (encode / decode round trip through the pipelined core, the fused GRU epilogue, the operand planes and the
    row-owned inverse kernel), and the batch is separable: the first 128 sequences alone give the same z (what batch
    sharding over GPUs relies on)."""
    hp, m = _model("bf16x3")
    m.eval()
    batch = to_device(kat_batch(hp, 256, 80, seed=12), DEV)
    with torch.no_grad():
        z_seq, loss, losses = m(batch)
        rec, _ = m.invert(z_seq, batch)
        half = {k: v[:128].contiguous() for k, v in batch.items()}
        z_half, _, nll_half = m(half)
    x = batch["p1_face"][:, 24:].transpose(0, 1)
    assert relerr(torch.stack(rec), x) < 5e-4
    assert relerr(torch.stack(z_half), torch.stack(z_seq)[:, :128]) < 1e-5
    assert relerr(torch.stack(nll_half), torch.stack(losses)[:, :128]) < 1e-5
    assert torch.isfinite(loss).all()


@pytest.mark.parametrize("mode,tol", [("bf16x3", 1e-4), ("bf16", 5e-3)])
def test_tensor_core_sampler_matches_fp32_sampler(mode, tol):
    """Autoregressive sampling, 200 sequences (ragged tiles) x 40 frames, identical injected noise: per-frame tcgen05
    conditioning GEMMs + row-owned inverse kernel (tensor-core modes) against the fully in-kernel fp32 sampler."""
    hp, m = _model("fp32")
    hy = O.Hyper.from_hparams(hp)
    m.eval()
    B, Tg = 200, 40
    T = hy.start_ts + Tg
    data = to_device(kat_batch(hp, B, T, seed=13), DEV)
    data["p1_face"] = torch.zeros(B, hy.start_ts, hy.C, device=DEV)
    noise = (torch.randn(Tg, B, hy.C, generator=torch.Generator().manual_seed(3)) * 0.7).to(DEV)
    x32 = m.inference(T, data=data, noise=noise)
    from lets_face_it_b200 import _cabi as cabi

    m.gemm_mode = {"bf16x3": cabi.GEMM_BF16X3, "bf16": cabi.GEMM_BF16}[mode]
    xtc = m.inference(T, data=data, noise=noise)
    assert xtc.shape == (B, Tg, hy.C)
    assert relerr(xtc, x32) < tol
    # and against the CPU oracle on a slice of the batch (the oracle is O(minutes) at full size)
    P = {k: v.detach() for k, v in oracle_params_from(m).items()}
    sl = {k: v[:8].cpu() for k, v in data.items()}
    x_ref = O.seq_inference(P, hy, sl, T, noise=noise[:, :8].cpu())
    assert relerr(xtc[:8], x_ref) < tol


@pytest.mark.parametrize("mode,tol", [("bf16x3", 2e-5), ("bf16", 5e-3)])
@pytest.mark.parametrize("B", [256, 100])
def test_persistent_encoder_feature_encode_matches_per_step_launches(mode, tol, B):
    """Feature encoding on the persistent window-GRU forward kernel (enc_persist.cu: all 24 / 2 / 16 window steps of a
    128-window tile in one launch, state resident in shared memory, halves exchanged through DSMEM; LFI_ENC_PERSIST_SAMPLE=1,
    the sampling default) against the chain of per-step launches (LFI_ENC_PERSIST_SAMPLE=0, the path training runs): encoded
    features.  Frame-dropout masks on.  B=100 leaves a ragged last tile (5,600 rows = 43.75 tiles)."""
    hp, m = _model(mode)
    hy = O.Hyper.from_hparams(hp)
    m.train()
    T = 80
    batch = to_device(kat_batch(hp, B, T, seed=31), DEV)
    masks = O.make_masks(hy, B, T - hy.start_ts, seed=32)
    m.injected_masks = {k: (v.to(DEV) if v is not None else None) for k, v in masks.items()}
    eng = m.engine()
    with _env(LFI_ENC_PERSIST_SAMPLE="1"):
        c1 = eng.feature_encode(batch, hy.start_ts, T - hy.start_ts, m.injected_masks).clone()
    with _env(LFI_ENC_PERSIST_SAMPLE="0"):
        c0 = eng.feature_encode(batch, hy.start_ts, T - hy.start_ts, m.injected_masks).clone()
    assert relerr(c1, c0) < tol
    # and the encoded features against the oracle on 8 sequences of the first two frames
    P = {k: v.detach() for k, v in oracle_params_from(m).items()}
    S = 8
    for ti in (0, 1):
        msl = {k: (v[:, :S].contiguous() if v is not None else None) for k, v in masks.items()}
        ref = O.conditioning(P, hy, {k: v[:S].cpu() for k, v in batch.items()}, hy.start_ts + ti, batch["p1_face"][:S].cpu(), msl, ti)
        got = eng.unfold_features(c1[ti * B: ti * B + S]).cpu()
        assert relerr(got, ref) < (1e-4 if mode == "bf16x3" else 5e-3)


@pytest.mark.parametrize("rnn", ["gru", "lstm"])
def test_wide_variant_matches_oracle(rnn):
    """BASELINE.json configs[4] shapes: 2x flow depth (K = 32), 2x hidden size (H = 256), GRU and LSTM coupling cells, in the
    bf16x3 and bf16 GEMM modes: forward z / NLL, the total gradient norm and per-tensor gradients against the oracle on the
    same inputs.  (Encoders and the time-parallel GEMMs run on the tcgen05 paths; the K = 32 / H = 256 flow core does not fit
    the stage-pipelined kernels and runs on the general wavefront kernels.)"""
    import copy

    from lets_face_it_b200 import _cabi as cabi

    hp = copy.deepcopy(final_hparams())
    hp.Glow["K"] = 32
    hp.Glow["hidden_channels"] = 256
    hp.Glow["rnn_type"] = rnn
    hy = O.Hyper.from_hparams(hp)
    m = build_kat_model(hp)
    m.glow.set_actnorm_init(True)
    P = O.clone_params(oracle_params_from(m), requires_grad=True)
    B, T = 64, 28
    batch = kat_batch(hp, B, T, seed=41)
    z_ref, nll_ref, loss_ref = O.seq_forward(P, hy, batch)
    loss_ref.backward()
    gr = torch.sqrt(sum((v.grad.double() ** 2).sum() for v in P.values() if v.grad is not None)).item()
    m = m.to(DEV).train()
    for mode, ztol, gtol in (("bf16x3", 1e-4, 1e-2), ("bf16", 5e-3, 0.15)):  # (twice the flow depth of final_model.yaml: 2x its 5e-3 bound)
        m.gemm_mode = {"bf16x3": cabi.GEMM_BF16X3, "bf16": cabi.GEMM_BF16}[mode]
        z, nll, g = _fwd_bwd(m, to_device(batch, DEV))
        assert relerr(z, z_ref.detach()) < ztol, mode
        assert relerr(nll, nll_ref.detach()) < 1e-4, mode
        gn = torch.sqrt(sum((v.double() ** 2).sum() for v in g.values())).item()
        assert abs(gn - gr) < (3e-3 if mode == "bf16x3" else 8e-2) * gr, (mode, gn, gr)
        worst = 0.0
        for n, v in g.items():
            ref = P[n].grad.double()
            worst = max(worst, float((v.double().cpu().reshape(ref.shape) - ref).norm() / ref.norm().clamp_min(1e-30)))
        assert worst < gtol, (mode, worst)


@pytest.mark.parametrize("rnn,H,K,B", [("lstm", 64, 3, 40), ("gru", 192, 5, 70)])
def test_hybrid_wavefronts_match_ffma_wavefronts_and_oracle(rnn, H, K, B):
    """Shapes outside the stage pipelines (LSTM, H != 128) in the tensor-core modes: the recurrent products of every wavefront
    run as ONE batched tcgen05 GEMM (forward h W_hh^T, backward dA_h W_hh) and the cell kernels skip them (LFI_WAVE_TC=1, the
    default) - against the all-FFMA wavefront kernels (LFI_WAVE_TC=0) and the oracle.  Ragged batches (B not a multiple of the
    128-row GEMM tile or of the cell tile)."""
    import copy

    from lets_face_it_b200 import _cabi as cabi

    hp = copy.deepcopy(final_hparams())
    hp.Glow["K"] = K
    hp.Glow["hidden_channels"] = H
    hp.Glow["rnn_type"] = rnn
    hy = O.Hyper.from_hparams(hp)
    m = build_kat_model(hp)
    m.glow.set_actnorm_init(True)
    P = O.clone_params(oracle_params_from(m), requires_grad=True)
    T = 30
    batch = kat_batch(hp, B, T, seed=43)
    z_ref, nll_ref, loss_ref = O.seq_forward(P, hy, batch)
    loss_ref.backward()
    m = m.to(DEV).train()
    m.gemm_mode = cabi.GEMM_BF16X3
    dbatch = to_device(batch, DEV)
    z1, n1, g1 = _fwd_bwd(m, dbatch)
    with _env(LFI_WAVE_TC="0"):
        z0, n0, g0 = _fwd_bwd(m, dbatch)
    assert relerr(z1, z0) < 2e-5 and relerr(n1, n0) < 1e-5
    assert relerr(z1, z_ref.detach()) < 1e-4 and relerr(n1, nll_ref.detach()) < 1e-4
    for k_ in g0:
        ref = g0[k_].double()
        err = float((g1[k_].double() - ref).norm() / ref.norm().clamp_min(1e-30))
        assert err < 2e-3, (k_, err)
        oref = P[k_].grad.double()
        oerr = float((g1[k_].double().cpu().reshape(oref.shape) - oref).norm() / oref.norm().clamp_min(1e-30))
        assert oerr < 5e-3, (k_, oerr)


@pytest.mark.parametrize("mode,tol", [("bf16x3", 2e-5), ("bf16", 5e-3)])
@pytest.mark.parametrize("B", [256, 100])
def test_input_projection_inside_the_step_gemm_matches_separate_projection(mode, tol, B):
    """Encoder window steps with the input projection inside the fused step GEMM (LFI_FUSE_GRU_FWD_X: masked window-input planes x
    W_ih as an extra k-block, step 0 = the input part alone; LFI_ENC_XFUSE=1, the default) against the same steps fetching the rows
    of a separate per-frame projection GEMM in the epilogue (LFI_ENC_XFUSE=0): z / NLL and every gradient (the backward pass reads
    the window-input planes the FORWARD pass gathered).  Frame-dropout masks on - the mask scales the A rows of the extra
    k-block instead of the projected rows.  B=100 leaves a ragged last tile."""
    hp, m = _model(mode)
    hy = O.Hyper.from_hparams(hp)
    m.train()
    T = 80
    batch = to_device(kat_batch(hp, B, T, seed=33), DEV)
    masks = O.make_masks(hy, B, T - hy.start_ts, seed=34)
    m.injected_masks = {k: (v.to(DEV) if v is not None else None) for k, v in masks.items()}
    with _env(LFI_ENC_XFUSE="1"):
        z1, n1, g1 = _fwd_bwd(m, batch)
    with _env(LFI_ENC_XFUSE="0"):
        z0, n0, g0 = _fwd_bwd(m, batch)
    assert relerr(z1, z0) < 5 * tol
    assert relerr(n1, n0) < (1e-5 if mode == "bf16x3" else 1e-4)
    for k in g0:
        ref = g0[k].double()
        err = float((g1[k].double() - ref).norm() / ref.norm().clamp_min(1e-30))
        assert err < (2e-3 if mode == "bf16x3" else 0.1), (k, err)
