"""GPU: the conditioning encoders under autograd.  In the reference, FeatureEncoder and ModalityEncoder are plain torch modules
(models.py:12-145), so the per-frame loop of SeqGlow.forward (create_conditioning -> glow) trains them.  Each case here is checked
against the oracle (oracle.encode_modality / oracle.conditioning) differentiated by torch in CPU fp32.

Bounds, relative to the reference tensor's max magnitude: values 1e-5 and gradients 1e-4 in fp32 and bf16x3 mode; in bf16 mode
values 1e-2 (the window-GRU steps of that mode carry a bf16 product, DESIGN.md §5) and gradients 0.15 in per-tensor relative L2
(the DESIGN.md §5 gradient bound of that mode)."""
import pytest
import torch

from lets_face_it_b200 import _cabi
from oracle import glow_oracle as O
from tests.helpers import final_hparams, relerr, small_hparams
from tests.kat import build_kat_model, oracle_params_from

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
MODES = {"fp32": _cabi.GEMM_FP32, "bf16x3": _cabi.GEMM_BF16X3, "bf16": _cabi.GEMM_BF16}
GRU_ATTRS = ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0")


def _hp(case):
    return small_hparams("gru") if case == "small" else final_hparams()


def _rel_l2(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def _check_grad(got, ref, mode, what):
    if mode == "bf16":
        assert _rel_l2(got, ref) <= 0.15, (what, _rel_l2(got, ref))
    else:
        assert relerr(got, ref) <= 1e-4, (what, relerr(got, ref))


def _val_tol(mode):
    return 1e-2 if mode == "bf16" else 1e-5


def _masks(hy, B, Tp, seed):
    """Frame-dropout masks [Tp, B, hist] of every modality (dropout 0.3 where the yaml has none, so that every stream is masked)."""
    g = torch.Generator().manual_seed(seed)
    out = {}
    for m in O.MODALITIES:
        if hy.hist[m]:
            p = hy.dropout[m] or 0.3
            out[m] = (torch.rand(Tp, B, hy.hist[m], generator=g) >= p).float() / (1.0 - p)
    return out


def _oracle_leaves(model):
    return {k: (v.requires_grad_(True) if ".encoder.weight" in k or ".encoder.bias" in k else v) for k, v in O.clone_params(oracle_params_from(model)).items()}


# ------------------------------------------------------------------------------------------------ ModalityEncoder
@pytest.mark.parametrize("case,modality", [("small", "p2_face"), ("small", "p1_speech"), ("final", "p2_face"), ("final", "p1_speech"),
                                           ("final", "p1_face")])
@pytest.mark.parametrize("with_mask", [False, True])
def test_modality_encoder_values_and_gradients(case, modality, with_mask, monkeypatch):
    hp = _hp(case)
    hy = O.Hyper.from_hparams(hp)
    model = build_kat_model(hp)
    P = _oracle_leaves(model)
    B = 64 if case == "small" else 256
    h, d = hy.hist[modality], hy.in_dim[modality]
    g = torch.Generator().manual_seed(11)
    x = torch.randn(B, h, d, generator=g)
    mask = _masks(hy, B, 1, seed=12)[modality][0] if with_mask else None
    xr = x.clone().requires_grad_(True)
    ref = O.encode_modality(P, hy, modality, xr, mask)
    R = torch.randn(ref.shape, generator=g)
    (ref * R).sum().backward()

    enc = getattr(model.feature_encoder, modality + "_encoder").to(DEV)
    monkeypatch.setattr(enc, "draw_mask", lambda lead, dev: mask.to(dev) if mask is not None else None)
    xd = x.to(DEV).requires_grad_(True)
    out = enc(xd)
    with torch.no_grad():
        out_ng = enc(xd)
    assert torch.equal(out, out_ng)  # fp32: the same kernels with and without grad mode
    assert relerr(out, ref) <= 1e-5
    (out * R.to(DEV)).sum().backward()
    assert relerr(xd.grad, xr.grad) <= 1e-4
    pre = "feature_encoder.%s_encoder.encoder." % modality
    for a in GRU_ATTRS if hy.enc[modality] == "rnn" else ():
        assert relerr(getattr(enc.encoder, a).grad, P[pre + a].grad) <= 1e-4, a


# ------------------------------------------------------------------------------------------------ FeatureEncoder
def _conditioning_case(case, mode, with_masks, seed=21):
    hp = _hp(case)
    hy = O.Hyper.from_hparams(hp)
    model = build_kat_model(hp)
    P = _oracle_leaves(model)
    B = 64 if case == "small" else 256
    T = hy.start_ts + 1
    data = O.synthetic_batch(hy, B, T, seed=seed)
    masks = _masks(hy, B, 1, seed=seed + 1) if with_masks else None
    return hp, hy, model, P, B, T, data, masks


def _device_conditioning(model, hy, data, masks, mode, monkeypatch, grad=True):
    model = model.to(DEV)
    model.gemm_mode = MODES[mode]
    fe = model.feature_encoder
    monkeypatch.setattr(fe, "draw_masks", lambda lead, dev: {k: v.to(dev) for k, v in masks.items()} if masks else None)
    dd = {k: v.to(DEV).requires_grad_(grad) for k, v in data.items()}
    with torch.set_grad_enabled(grad):
        out = model.create_conditioning(dd, hy.start_ts, None, dd["p1_face"])
    return out, dd


@pytest.mark.parametrize("case,mode", [("small", "fp32"), ("final", "fp32"), ("final", "bf16x3"), ("final", "bf16")])
@pytest.mark.parametrize("with_masks", [False, True])
def test_feature_encoder_values_and_gradients(case, mode, with_masks, monkeypatch):
    hp, hy, model, P, B, T, data, masks = _conditioning_case(case, mode, with_masks)
    dr = {k: v.clone().requires_grad_(True) for k, v in data.items()}
    ref = O.conditioning(P, hy, dr, hy.start_ts, dr["p1_face"], masks, 0)
    R = torch.randn(ref.shape, generator=torch.Generator().manual_seed(5))
    (ref * R).sum().backward()

    out_ng, _ = _device_conditioning(model, hy, data, masks, mode, monkeypatch, grad=False)
    out, dd = _device_conditioning(model, hy, data, masks, mode, monkeypatch)
    assert out.requires_grad
    if mode == "fp32":
        assert torch.equal(out, out_ng)
    else:  # the no-grad call runs the persistent window-GRU kernel, the grad-mode call the training step's launches
        assert relerr(out, out_ng) <= _val_tol(mode)
    assert relerr(out, ref) <= _val_tol(mode), relerr(out, ref)
    (out * R.to(DEV)).sum().backward()
    for m in O.MODALITIES:
        if hy.hist[m]:
            _check_grad(dd[m].grad, dr[m].grad, mode, m)
    for m in O.MODALITIES:
        gru = model.feature_encoder.gru_of(m)
        if gru is None:
            continue
        for a in GRU_ATTRS:
            _check_grad(getattr(gru, a).grad, P["feature_encoder.%s_encoder.encoder.%s" % (m, a)].grad, mode, (m, a))


@pytest.mark.parametrize("mode", ["fp32", "bf16x3", "bf16"])
def test_feature_encoder_backward_is_bitwise_reproducible(mode, monkeypatch):
    hp, hy, model, P, B, T, data, masks = _conditioning_case("final", mode, True)
    R = None
    runs = []
    for _ in range(2):
        model.zero_grad(set_to_none=True)
        out, dd = _device_conditioning(model, hy, data, masks, mode, monkeypatch)
        if R is None:
            R = torch.randn(out.shape, generator=torch.Generator().manual_seed(6)).to(DEV)
        (out * R).sum().backward()
        grads = [dd[m].grad.clone() for m in O.MODALITIES if hy.hist[m]]
        grads += [p.grad.clone() for p in model.feature_encoder.gru_params()]
        runs.append((out.detach().clone(), grads))
    assert torch.equal(runs[0][0], runs[1][0])
    for a, b in zip(runs[0][1], runs[1][1]):
        assert torch.equal(a, b)


# ------------------------------------------------------------------------------------------------ C ABI, overlapping windows
@pytest.mark.parametrize("case,mode", [("small", "fp32"), ("final", "bf16x3")])
def test_cabi_overlapping_windows(case, mode):
    """Tp = 3 frames in one call: the windows of neighbouring frames overlap, so dx of a frame sums several windows."""
    hp = _hp(case)
    hy = O.Hyper.from_hparams(hp)
    model = build_kat_model(hp)
    P = _oracle_leaves(model)
    B, Tp = (32, 3) if case == "small" else (128, 3)
    T = hy.start_ts + Tp + 1
    data = O.synthetic_batch(hy, B, T, seed=31)
    masks = _masks(hy, B, Tp, seed=32)
    t0 = hy.start_ts + 1  # not the first frame: the last frame of the batch is read by no window but the p1_face ones do not
    dr = {k: v.clone().requires_grad_(True) for k, v in data.items()}
    g = torch.Generator().manual_seed(33)
    Rs = [torch.randn(B, hy.F, generator=g) for _ in range(Tp)]
    loss = sum((O.conditioning(P, hy, dr, t0 + i, dr["p1_face"], masks, i) * Rs[i]).sum() for i in range(Tp))
    loss.backward()

    model = model.to(DEV)
    model.gemm_mode = MODES[mode]
    eng = model.engine()
    dmasks = {k: v.to(DEV) for k, v in masks.items()}
    dd = {k: v.to(DEV) for k, v in data.items()}
    cond, saved = eng.feature_encode_train(dd, t0, Tp, dmasks)
    with torch.no_grad():
        ref_fold = eng.feature_encode(dd, t0, Tp, dmasks)
    assert relerr(cond, ref_fold) <= _val_tol(mode)
    # dL/d(folded cond): the adjoint of unfold_features sums the two copies of a GRU state
    ph = torch.zeros_like(cond, requires_grad=True)
    R = torch.cat(Rs, dim=0).to(DEV)
    (eng.unfold_features(ph) * R).sum().backward()
    dx, grads = eng.feature_encode_backward(saved, ph.grad, [True] * 4)
    for i, m in enumerate(O.MODALITIES):
        if hy.hist[m]:
            _check_grad(dx[i], dr[m].grad, mode, m)
        if grads[i] is not None:
            for a, t in zip(GRU_ATTRS, grads[i]):
                _check_grad(t, P["feature_encoder.%s_encoder.encoder.%s" % (m, a)].grad, mode, (m, a))
    if hy.hist["p2_speech"] and hy.hist["p2_speech"] < hy.start_ts:  # frames before every window: exactly zero
        first = t0 - hy.hist["p2_speech"] + 1
        assert bool((dx[3][:, :first] == 0).all())


# ------------------------------------------------------------------------------------------------ end to end
def test_per_frame_training_loop_matches_seqglow_forward():
    """The reference's SeqGlow.forward loop written with the public modules (create_conditioning -> glow -> NLL per frame) gives
    every parameter, feature_encoder.* included, the gradient SeqGlow.forward(batch)[1].backward() gives."""
    hp = small_hparams("gru")
    hy = O.Hyper.from_hparams(hp)
    m = build_kat_model(hp, DEV).train()
    m.glow.set_actnorm_init(True)
    B, Tp = 24, 4
    T = hy.start_ts + Tp
    batch = {k: v.to(DEV) for k, v in O.synthetic_batch(hy, B, T, seed=41).items()}

    m.glow.init_rnn_hidden()
    total = 0.0
    for t in range(hy.start_ts, T):
        cond = m.create_conditioning(batch, t, None, batch["p1_face"])
        z, logdet = m.glow(x=batch["p1_face"][:, t, :], condition=cond)
        total = total + m.loss(logdet.clone(), z).mean()  # (SeqGlow.loss adds to its first argument in place)
    (total / Tp).backward()
    loop = {n: p.grad.detach().clone() for n, p in m.named_parameters()}
    m.zero_grad(set_to_none=True)
    _, loss, _ = m(batch)
    loss.backward()
    fused = {n: p.grad.detach().clone() for n, p in m.named_parameters()}
    assert any(".encoder." in n for n in loop)
    for n, g in loop.items():
        assert g is not None and fused[n] is not None, n
        assert _rel_l2(g, fused[n]) <= 1e-4, (n, _rel_l2(g, fused[n]))
