"""GPU: SeqGlow.forward differentiated with respect to its batch.  In the reference, SeqGlow.forward is plain torch (models.py:534-561),
so batch tensors that require grad get dL/d(stream) from loss.backward(); here the streams enter the fused node and
lfi_seq_train_bwd_dx returns their gradients.  Every case is checked against oracle.seq_forward differentiated by torch in CPU fp32,
with every stream requiring grad, with and without frame-dropout masks on every stream.

  * small shapes (GRU / LSTM, affine / additive): fp32 runs the wavefront backward, bf16x3 the hybrid wavefronts;
  * final_model.yaml at B = 256, T = 80: fp32 runs the FFMA stage pipeline, bf16x3 and bf16 the tcgen05 stage pipeline, and bf16x3
    once more with LFI_CORE_TC_BWD=0 (FFMA pipeline in a tensor-core mode).  The loss is restricted to the first 16 sequences
    (d nll zero elsewhere, as in test_gpu_pinned.py), so the input gradients of the other 240 must be exactly zero.

Bounds (DESIGN.md section 5 gradient bounds): fp32 max|err| <= 1e-4 max|ref|; bf16x3 <= 5e-3 and bf16 <= 0.15 per-tensor relative L2.
Frames that no window and no flow input reads are exact zeros, in the oracle too.  In the same call, z and the NLL are bitwise
those of the same model without input gradients, and the parameter gradients agree to 1e-6 relative L2 in fp32 (reduction order
only) and to 1e-3 in the tensor-core modes, whose training backward is not run-to-run reproducible by itself."""
import pytest
import torch

from lets_face_it_b200 import _cabi
from oracle import glow_oracle as O
from tests.helpers import final_hparams, relerr, small_hparams
from tests.kat import build_kat_model, kat_batch, oracle_params_from

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
MODES = {"fp32": _cabi.GEMM_FP32, "bf16x3": _cabi.GEMM_BF16X3, "bf16": _cabi.GEMM_BF16}
RESULTS = {}  # measured errors, printed by the last test (pytest -s)


def _rel_l2(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def _err(got, ref, mode):
    return relerr(got, ref) if mode == "fp32" else _rel_l2(got, ref)


def _bound(mode):
    return {"fp32": 1e-4, "bf16x3": 5e-3, "bf16": 0.15}[mode]


def _masks(hy, B, Tp, seed):
    """Frame-dropout masks [Tp, B, hist] of every stream (dropout 0.3 where the yaml has none)."""
    g = torch.Generator().manual_seed(seed)
    out = {}
    for m in O.MODALITIES:
        if hy.hist[m]:
            p = hy.dropout[m] or 0.3
            out[m] = (torch.rand(Tp, B, hy.hist[m], generator=g) >= p).float() / (1.0 - p)
    return out


def _first_read(hy, m):
    """First frame any window or the flow input reads (p1_face's window ends before frame t)."""
    return hy.start_ts - hy.hist[m] if m == "p1_face" else hy.start_ts - hy.hist[m] + 1


_ORACLE = {}


def _oracle(key, P, hy, batch, masks, S):
    """dL/d(stream) of the oracle's loss over the first S sequences (cached: the modes share parameters and data)."""
    if key not in _ORACLE:
        sl = {k: v[:S].clone().requires_grad_(True) for k, v in batch.items()}
        msl = {k: v[:, :S].contiguous() for k, v in masks.items()} if masks else None
        _, _, loss = O.seq_forward({k: v.detach().clone().requires_grad_(v.requires_grad) for k, v in P.items()}, hy, sl, msl)
        loss.backward()
        _ORACLE[key] = {k: v.grad for k, v in sl.items() if hy.hist[k]}
    return _ORACLE[key]


def _seqglow_node(loss):
    seen, stack = set(), [loss.grad_fn]
    while stack:
        n = stack.pop()
        if n is None or n in seen:
            continue
        seen.add(n)
        if "_SeqGlowFn" in n.name():
            return n
        stack.extend(f for f, _ in n.next_functions)
    raise AssertionError("no SeqGlow node in the graph")


def _forward_backward(m, batch, S):
    """SeqGlow.forward -> loss.backward(), with d nll of the sequences >= S set to zero (and the rest scaled to a mean over S)."""
    z_seq, loss, losses = m(batch)
    B = z_seq[0].shape[0]

    def pre(grads):
        dz, dnll = grads
        d = dnll.clone()
        d[:, S:] = 0
        return dz, d * (B / S)

    _seqglow_node(loss).register_prehook(pre)
    loss.backward()
    torch.cuda.synchronize()
    return torch.stack(z_seq), torch.stack(losses)


def _run_case(tag, hp, mode, B, T, S, masked, seed=31):
    hy = O.Hyper.from_hparams(hp)
    Tp = T - hy.start_ts
    m = build_kat_model(hp)
    m.glow.set_actnorm_init(True)
    P = O.clone_params(oracle_params_from(m), requires_grad=True)
    batch = kat_batch(hp, B, T, seed=seed)
    masks = _masks(hy, B, Tp, seed + 1) if masked else None
    ref = _oracle((tag, masked), P, hy, batch, masks, S)

    m = m.to(DEV).train()
    m.gemm_mode = MODES[mode]
    if masked:
        m.injected_masks = {k: v.to(DEV) for k, v in masks.items()}
    dbatch = {k: v.to(DEV) for k, v in batch.items()}
    z0, nll0 = _forward_backward(m, dbatch, S)
    pg0 = {n: p.grad.detach().clone() for n, p in m.named_parameters()}
    m.zero_grad(set_to_none=True)
    xs = {k: v.clone().requires_grad_(True) for k, v in dbatch.items()}
    z1, nll1 = _forward_backward(m, xs, S)

    assert torch.equal(z0, z1) and torch.equal(nll0, nll1)
    # fp32: reduction order only.  The tensor-core modes' training backward varies from run to run by itself (split-K atomics
    # feeding bf16 operand planes; measured up to 1e-4 on the p2_face encoder's weight_ih between two plain calls).
    pbound = 1e-6 if mode == "fp32" else 1e-3
    for n, p in m.named_parameters():
        assert _rel_l2(p.grad, pg0[n]) <= pbound, (n, _rel_l2(p.grad, pg0[n]))
    errs = {}
    for k in O.MODALITIES:
        if not hy.hist[k]:
            assert xs[k].grad is None or not bool(xs[k].grad.any())
            continue
        g = xs[k].grad
        assert g is not None and g.shape == (B, T, hy.in_dim[k]), k
        assert bool((g[S:] == 0).all()), k  # sequences outside the loss
        f0 = _first_read(hy, k)
        assert bool((g[:, :f0] == 0).all()) and bool((ref[k][:, :f0] == 0).all()), k  # frames nothing reads
        errs[k] = _err(g[:S], ref[k], mode)
        assert errs[k] <= _bound(mode), (k, errs[k])
    RESULTS["%s %s masks=%s" % (tag, mode, masked)] = errs


@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("mode", ["fp32", "bf16x3"])
@pytest.mark.parametrize("rnn,coupling", [("gru", "affine"), ("lstm", "affine"), ("gru", "additive")])
def test_small_shapes_against_oracle(rnn, coupling, mode, masked):
    hp = small_hparams(rnn)
    hp.Glow["flow_coupling"] = coupling
    hy = O.Hyper.from_hparams(hp)
    _run_case("small-%s-%s" % (rnn, coupling), hp, mode, 32, hy.start_ts + 6, 32, masked)


@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("mode,tc_bwd", [("fp32", True), ("bf16x3", True), ("bf16", True), ("bf16x3", False)])
def test_final_model_against_oracle_slice(mode, tc_bwd, masked, monkeypatch):
    if not tc_bwd:
        monkeypatch.setenv("LFI_CORE_TC_BWD", "0")
    _run_case("final", final_hparams(), mode, 256, 80, 16, masked)


def test_launches_unchanged_without_input_grads():
    """No batch tensor requires grad: SeqGlow.forward + loss.backward() launch exactly the kernels of a plain
    lfi_seq_train_fwd + lfi_seq_train_bwd pair; with input gradients there are more."""
    hp = final_hparams()
    hy = O.Hyper.from_hparams(hp)
    L = _cabi.lib()
    m = build_kat_model(hp, DEV).train()
    m.glow.set_actnorm_init(True)
    m.gemm_mode = _cabi.GEMM_BF16X3
    B, T = 256, 80
    batch = {k: v.to(DEV) for k, v in kat_batch(hp, B, T, seed=5).items()}
    masks = {k: v.to(DEV) for k, v in _masks(hy, B, T - hy.start_ts, 6).items()}
    m.injected_masks = masks

    def count(fn):
        torch.cuda.synchronize()
        n0 = L.lfi_launch_count()
        fn()
        torch.cuda.synchronize()
        return L.lfi_launch_count() - n0

    def module(b):
        _, loss, _ = m(b)
        loss.backward()

    def engine():
        eng = m.engine()
        z, nll = eng.train_forward(batch, masks)
        eng.train_backward(z, torch.full_like(nll, 1.0 / nll.numel()), eng.new_flat_grad())

    module(batch)  # warm-up
    n_module, n_engine = count(lambda: module(batch)), count(engine)
    assert n_module == n_engine, (n_module, n_engine)
    n_dx = count(lambda: module({k: v.clone().requires_grad_(True) for k, v in batch.items()}))
    assert n_dx > n_module
    with torch.no_grad():  # grad mode off: the streams are not inputs of the node, nothing extra runs
        n_nograd_fwd = count(lambda: m({k: v.clone().requires_grad_(True) for k, v in batch.items()}))
        n_plain_fwd = count(lambda: m(batch))
    assert n_nograd_fwd == n_plain_fwd


def test_per_frame_loop_matches_seqglow_forward():
    """The reference's SeqGlow.forward loop written with the public modules (create_conditioning -> glow -> NLL per frame) gives
    every stream the gradient SeqGlow.forward(batch)[1].backward() gives (fp32 mode)."""
    hp = small_hparams("gru")
    hy = O.Hyper.from_hparams(hp)
    m = build_kat_model(hp, DEV).train()
    m.glow.set_actnorm_init(True)
    B, Tp = 24, 4
    T = hy.start_ts + Tp
    base = {k: v.to(DEV) for k, v in O.synthetic_batch(hy, B, T, seed=41).items()}

    batch = {k: v.clone().requires_grad_(True) for k, v in base.items()}
    m.glow.init_rnn_hidden()
    total = 0.0
    for t in range(hy.start_ts, T):
        cond = m.create_conditioning(batch, t, None, batch["p1_face"])
        z, logdet = m.glow(x=batch["p1_face"][:, t, :], condition=cond)
        total = total + m.loss(logdet.clone(), z).mean()  # (SeqGlow.loss adds to its first argument in place)
    (total / Tp).backward()
    loop = {k: v.grad.detach().clone() for k, v in batch.items() if hy.hist[k]}

    fused_in = {k: v.clone().requires_grad_(True) for k, v in base.items()}
    _, loss, _ = m(fused_in)
    loss.backward()
    errs = {}
    for k, g in loop.items():
        errs[k] = relerr(fused_in[k].grad, g)
        assert errs[k] <= 1e-4, (k, errs[k])
    RESULTS["per-frame loop vs fused fp32"] = errs


def test_zz_report():
    for k, v in RESULTS.items():
        print("input-gradient error", k, {m: "%.2e" % e for m, e in v.items()})
