"""GPU: the stand-alone modules under autograd.  In the reference, ActNorm2d, InvertibleConv1x1, LinearZeros and f_seq are plain
torch modules (modules.py:45-95, 122-194; models.py:148-214), so a user who trains one of them on its own gets gradients.
Each case here is checked against the oracle restatement (oracle/glow_oracle.py) differentiated by torch in CPU fp32."""
import types

import numpy as np
import pytest
import torch

from oracle import glow_oracle as O
from tests.helpers import relerr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _leaf(t):
    return t.detach().clone().float().requires_grad_(True)


def _dev_leaf(t):
    return t.detach().to(DEV).requires_grad_(True)


def _logdet_arg(kind, B, device):
    if kind == "none":
        return None
    if kind == "zero":
        return 0
    return torch.linspace(-1.0, 1.0, B).to(device)


def _loss(y, ld, Ry, Rl):
    loss = (y * Ry).sum()
    if ld is not None:
        loss = loss + (ld * Rl).sum()
    return loss


# ------------------------------------------------------------------------------------------------ ActNorm2d
@pytest.mark.parametrize("reverse", [False, True])
@pytest.mark.parametrize("logdet", ["none", "zero", "tensor"])
def test_actnorm_values_and_gradients(reverse, logdet):
    from lets_face_it_b200.glow import ActNorm2d

    torch.manual_seed(1)
    B, C = 21, 13
    m = ActNorm2d(C)
    with torch.no_grad():
        m.bias.copy_(torch.randn(1, C) * 0.3)
        m.logs.copy_(torch.randn(1, C) * 0.3)
    m.inited = True
    x = torch.randn(B, C)
    Ry, Rl = torch.randn(B, C), torch.randn(B)
    P = {"a.bias": _leaf(m.bias), "a.logs": _leaf(m.logs)}
    xr = _leaf(x)
    y_ref, ld_ref = O.actnorm(P, "a.", xr, _logdet_arg(logdet, B, "cpu"), reverse)
    _loss(y_ref, ld_ref, Ry, Rl).backward()

    m = m.to(DEV)
    xd = _dev_leaf(x)
    y, ld = m(xd, _logdet_arg(logdet, B, DEV), reverse)
    assert relerr(y, y_ref) <= 1e-6
    if logdet == "none":
        assert ld is None
    else:
        assert relerr(ld, ld_ref) <= 1e-6
    _loss(y, ld, Ry.to(DEV), Rl.to(DEV)).backward()
    assert relerr(xd.grad, xr.grad) <= 1e-5
    assert relerr(m.bias.grad, P["a.bias"].grad) <= 1e-5
    assert relerr(m.logs.grad, P["a.logs"].grad) <= 1e-5


# ------------------------------------------------------------------------------------------------ InvertibleConv1x1
def _invconv_case(C, LU, seed):
    from lets_face_it_b200.glow import InvertibleConv1x1

    np.random.seed(seed)
    torch.manual_seed(seed)
    m = InvertibleConv1x1(C, LU_decomposed=LU)
    if LU:
        with torch.no_grad():  # off the identity-like init, so that every entry of L and U matters
            m.l.add_(0.05 * torch.randn(C, C))
            m.u.add_(0.05 * torch.randn(C, C))
            m.log_s.add_(0.1 * torch.randn(C))
    else:
        with torch.no_grad():  # off the orthogonal init, whose log|det W| = 0 would make the log-det term all rounding
            m.weight.add_(0.1 * torch.randn(C, C))
    P = {"c." + k: (_leaf(v) if k in ("l", "u", "log_s", "weight") else v.detach().clone().float()) for k, v in m.state_dict().items()}
    return m, P


@pytest.mark.parametrize("C", [56, 7])
@pytest.mark.parametrize("LU", [True, False])
@pytest.mark.parametrize("reverse", [False, True])
def test_invconv_values_and_gradients(C, LU, reverse):
    m, P = _invconv_case(C, LU, seed=5 + C)
    B = 33
    x = torch.randn(B, C)
    Ry, Rl = torch.randn(B, C), torch.randn(B)
    xr = _leaf(x)
    z_ref, ld_ref = O.invconv(P, "c.", xr, torch.zeros(B), reverse, LU)
    _loss(z_ref, ld_ref, Ry, Rl).backward()

    m = m.to(DEV)
    xd = _dev_leaf(x)
    z, ld = m(xd, torch.zeros(B, device=DEV), reverse)
    assert relerr(z, z_ref) <= (1e-4 if reverse else 1e-5)
    assert relerr(ld, ld_ref) <= 1e-5
    _loss(z, ld, Ry.to(DEV), Rl.to(DEV)).backward()
    assert relerr(xd.grad, xr.grad) <= 1e-4
    names = ("l", "u", "log_s") if LU else ("weight",)
    for n in names:
        assert relerr(getattr(m, n).grad, P["c." + n].grad) <= 1e-4, n
    if LU:
        lower = torch.tril(torch.ones(C, C, dtype=torch.bool, device=DEV), -1)
        assert bool((m.l.grad[~lower] == 0).all())
        assert bool((m.u.grad[~lower.t()] == 0).all())


@pytest.mark.parametrize("LU", [True, False])
@pytest.mark.parametrize("reverse", [False, True])
def test_invconv_get_weight_alone_is_differentiable(LU, reverse):
    C = 7
    m, P = _invconv_case(C, LU, seed=11)
    R = torch.randn(C, C)
    w_ref, _ = O.invconv_weight(P, "c.", C, reverse, LU)
    (w_ref * R).sum().backward()
    m = m.to(DEV)
    w, _ = m.get_weight(torch.zeros(2, C, device=DEV), reverse)
    assert w.requires_grad
    assert relerr(w, w_ref) <= 1e-5
    (w * R.to(DEV)).sum().backward()
    for n in (("l", "u", "log_s") if LU else ("weight",)):
        assert relerr(getattr(m, n).grad, P["c." + n].grad) <= 1e-4, n


# ------------------------------------------------------------------------------------------------ LinearZeros
@pytest.mark.parametrize("perturbed", [False, True])
def test_linear_zeros_values_and_gradients(perturbed):
    from lets_face_it_b200.glow import LinearZeros

    torch.manual_seed(2)
    B, In, Out = 21, 20, 7
    m = LinearZeros(In, Out)
    if perturbed:
        with torch.no_grad():
            m.weight.normal_(0, 0.2)
            m.bias.normal_(0, 0.2)
            m.logs.normal_(0, 0.1)
    P = {"f." + k: _leaf(v) for k, v in m.state_dict().items()}
    x = torch.randn(B, In)
    R = torch.randn(B, Out)
    xr = _leaf(x)
    out_ref = O.linear_zeros(P, "f.", xr)
    (out_ref * R).sum().backward()

    m = m.to(DEV)
    xd = _dev_leaf(x)
    out = m(xd)
    assert relerr(out, out_ref) <= 1e-5
    (out * R.to(DEV)).sum().backward()
    assert relerr(xd.grad, xr.grad) <= 1e-4
    for n in ("weight", "bias", "logs"):
        assert relerr(getattr(m, n).grad, P["f." + n].grad) <= 1e-4, n


# ------------------------------------------------------------------------------------------------ f_seq
FSEQ_SHAPES = {"odd": dict(In=7, Out=3, H=20, D=24, F=40, B=21), "final": dict(In=28, Out=56, H=128, D=512, F=1560, B=256)}
FSEQ_PARAMS = ("cond_transform.0.weight", "cond_transform.0.bias", "rnn.weight_ih", "rnn.bias_ih", "rnn.weight_hh", "rnn.bias_hh",
               "final_linear.weight", "final_linear.bias", "final_linear.logs")


def _fseq(rnn, s, seed=3):
    from lets_face_it_b200.glow import f_seq

    torch.manual_seed(seed)
    f = f_seq(s["In"], s["Out"], s["H"], s["D"], s["F"], rnn)
    with torch.no_grad():
        f.final_linear.weight.normal_(0, 0.1)
        f.final_linear.bias.normal_(0, 0.1)
        f.final_linear.logs.normal_(0, 0.1)
    return f


def _fseq_frames(s, T=3, seed=4):
    g = torch.Generator().manual_seed(seed)
    zs = [torch.randn(s["B"], s["In"], generator=g) for _ in range(T)]
    cs = [torch.randn(s["B"], s["F"], generator=g) for _ in range(T)]
    Rs = [torch.randn(s["B"], s["Out"], generator=g) for _ in range(T)]
    return zs, cs, Rs


def _fseq_device_run(f, zs, cs, Rs):
    f.init_rnn_hidden()
    zd = [_dev_leaf(z) for z in zs]
    cd = [_dev_leaf(c) for c in cs]
    outs = [f(z, c) for z, c in zip(zd, cd)]
    loss = sum((o * R.to(DEV)).sum() for o, R in zip(outs, Rs))
    f.zero_grad()
    loss.backward()
    return outs, zd, cd


@pytest.mark.parametrize("shape", ["odd", "final"])
@pytest.mark.parametrize("rnn", ["gru", "lstm"])
def test_fseq_three_frames_match_oracle(rnn, shape):
    s = FSEQ_SHAPES[shape]
    f = _fseq(rnn, s)
    zs, cs, Rs = _fseq_frames(s)
    P = {"f." + k: _leaf(v) for k, v in f.state_dict().items()}
    hy = types.SimpleNamespace(rnn_type=rnn, H=s["H"])
    zr, cr = [_leaf(z) for z in zs], [_leaf(c) for c in cs]
    state = {}
    outs_ref = [O.coupling_net(P, "f.", hy, z, c, state, 0) for z, c in zip(zr, cr)]
    sum((o * R).sum() for o, R in zip(outs_ref, Rs)).backward()

    f = f.to(DEV)
    outs, zd, cd = _fseq_device_run(f, zs, cs, Rs)
    h_ref = state[0] if rnn == "gru" else state[0][0]
    assert f.hidden.shape == (s["B"], s["H"]) and relerr(f.hidden, h_ref) <= 1e-5
    if rnn == "lstm":
        assert relerr(f.cell, state[0][1]) <= 1e-5
    for o, r in zip(outs, outs_ref):
        assert relerr(o, r) <= 1e-5
    for a, b in zip(zd + cd, zr + cr):
        assert relerr(a.grad, b.grad) <= 1e-4
    sd = dict(f.named_parameters())
    for n in FSEQ_PARAMS:
        assert relerr(sd[n].grad, P["f." + n].grad) <= 1e-4, n


# ------------------------------------------------------------------------------------------------ determinism, grad mode
@pytest.mark.parametrize("rnn", ["gru", "lstm"])
def test_backward_is_bitwise_deterministic(rnn):
    """Two identical backward calls give bitwise-equal gradients (fixed-order reductions, no split-K atomics); B is large
    enough that the row reductions are long."""
    from lets_face_it_b200.glow import ActNorm2d, LinearZeros

    s = dict(FSEQ_SHAPES["final"], B=2048)
    f = _fseq(rnn, s).to(DEV)
    zs, cs, Rs = _fseq_frames(s, T=2)
    grads = []
    for _ in range(2):
        _fseq_device_run(f, zs, cs, Rs)
        grads.append([p.grad.clone() for p in f.parameters()])
    assert all(torch.equal(a, b) for a, b in zip(*grads))

    torch.manual_seed(6)
    an, lz = ActNorm2d(37).to(DEV), LinearZeros(30, 11).to(DEV)
    an.inited = True
    with torch.no_grad():
        lz.weight.normal_(0, 0.2)
        lz.logs.normal_(0, 0.1)
    x, h = torch.randn(4099, 37, device=DEV), torch.randn(4099, 30, device=DEV)
    R1, R2 = torch.randn(4099, 37, device=DEV), torch.randn(4099, 11, device=DEV)
    grads = []
    for _ in range(2):
        an.zero_grad()
        lz.zero_grad()
        y, _ = an(x, None, False)
        ((y * R1).sum() + (lz(h) * R2).sum()).backward()
        grads.append([p.grad.clone() for p in list(an.parameters()) + list(lz.parameters())])
    assert all(torch.equal(a, b) for a, b in zip(*grads))


def test_forward_values_do_not_depend_on_grad_mode():
    from lets_face_it_b200.glow import ActNorm2d, InvertibleConv1x1, LinearZeros

    torch.manual_seed(7)
    np.random.seed(7)
    B = 19
    an = ActNorm2d(9).to(DEV)
    an.inited = True
    with torch.no_grad():
        an.logs.normal_(0, 0.3)
    lz = LinearZeros(9, 5).to(DEV)
    with torch.no_grad():
        lz.weight.normal_(0, 0.3)
    x = torch.randn(B, 9, device=DEV)
    cases = [lambda: an(x, torch.zeros(B, device=DEV), False), lambda: an(x, 0, True), lambda: (lz(x),)]
    for LU in (True, False):
        conv = InvertibleConv1x1(9, LU_decomposed=LU).to(DEV)
        cases += [lambda c=conv: c(x, torch.zeros(B, device=DEV), False), lambda c=conv: c(x, 0, True)]
    for fn in cases:
        with torch.no_grad():
            ref = fn()
        got = fn()
        assert got[0].requires_grad
        for a, b in zip(got, ref):
            if torch.is_tensor(a):
                assert torch.equal(a, b)
    for rnn in ("gru", "lstm"):
        s = FSEQ_SHAPES["odd"]
        f = _fseq(rnn, s).to(DEV)
        zs, cs, _ = _fseq_frames(s)
        zs, cs = [z.to(DEV) for z in zs], [c.to(DEV) for c in cs]
        res = []
        for grad in (False, True):
            f.init_rnn_hidden()
            with torch.set_grad_enabled(grad):
                res.append([(f(z, c), f.hidden, f.cell) for z, c in zip(zs, cs)])
        for (o0, h0, c0), (o1, h1, c1) in zip(*res):
            assert o1.requires_grad and torch.equal(o0, o1) and torch.equal(h0, h1)
            assert (c0 is None and c1 is None) if rnn == "gru" else torch.equal(c0, c1)


# ------------------------------------------------------------------------------------------------ interop with FlowStep
def _hyper(C, H, D, rnn):
    return O.Hyper(C=C, K=1, H=H, D=D, rnn_type=rnn, scale_eps=1e-4, actnorm_scale=1.0, LU=True, coupling="affine",
                   hist={m: 1 for m in O.MODALITIES}, enc={m: "none" for m in O.MODALITIES}, enc_hidden={m: 0 for m in O.MODALITIES},
                   in_dim={m: 1 for m in O.MODALITIES}, dropout={m: 0.0 for m in O.MODALITIES})


@pytest.mark.parametrize("rnn", ["gru", "lstm"])
def test_fseq_state_feeds_flowstep(rnn):
    """f_seq.forward on the coupling network of a FlowStep whose engine exists (its parameters are views into the flat
    buffer), then FlowStep.forward on the same step: the step reads the state f_seq left behind, and values and gradients
    (through that state, back to f_seq's inputs) match the oracle."""
    from lets_face_it_b200.glow import FlowStep

    np.random.seed(8)
    torch.manual_seed(8)
    C, H, D, Fr, B = 12, 16, 24, 40, 21
    step = FlowStep(C, H, D, flow_permutation="invconv", flow_coupling="affine", LU_decomposed=True, scale_eps=1e-4,
                    feature_encoder_dim=Fr, glow_rnn_type=rnn)
    with torch.no_grad():
        for n, p in step.named_parameters():
            if "final_linear" in n or "actnorm" in n:
                p.normal_(0, 0.15)
    step.actnorm.inited = True
    hy = _hyper(C, H, D, rnn)
    P = O.clone_params({"glow.flow.layers.0." + k: v for k, v in step.state_dict().items()}, requires_grad=True)
    z1, c0, x, c1 = torch.randn(B, C // 2), torch.randn(B, Fr), torch.randn(B, C), torch.randn(B, Fr)
    R0, R1, Rl = torch.randn(B, C), torch.randn(B, C), torch.randn(B)
    leaves = [_leaf(t) for t in (z1, c0, x, c1)]
    state = {}
    h = O.coupling_net(P, "glow.flow.layers.0.f.", hy, leaves[0], leaves[1], state, 0)
    y, ld = O.flow_step(P, hy, 0, leaves[2], leaves[3], torch.zeros(B), False, state)
    ((h * R0).sum() + (y * R1).sum() + (ld * Rl).sum()).backward()

    step = step.to(DEV)
    with torch.no_grad():
        step(x.to(DEV), c1.to(DEV), None, False)  # builds the engine: parameters become views into its flat buffer
    step.init_rnn_hidden()
    dl = [_dev_leaf(t) for t in (z1, c0, x, c1)]
    hd = step.f(dl[0], dl[1])
    yd, ldd = step(dl[2], dl[3], torch.zeros(B, device=DEV), False)
    assert relerr(hd, h) <= 1e-5
    assert relerr(yd, y) <= 1e-4 and relerr(ldd, ld) <= 1e-4
    ((hd * R0.to(DEV)).sum() + (yd * R1.to(DEV)).sum() + (ldd * Rl.to(DEV)).sum()).backward()
    for a, b in zip(dl, leaves):
        assert relerr(a.grad, b.grad) < 2e-3
    for n, p in step.named_parameters():
        assert p.grad is not None, n
        assert relerr(p.grad, P["glow.flow.layers.0." + n].grad) < 3e-3, n


# ------------------------------------------------------------------------------------------------ FlowNet.encode: one refresh per call
def test_flownet_encode_refreshes_once_under_autograd():
    """FlowNet.encode under autograd rebuilds the derived weight cache once per call, not once per step.  Outputs and the
    gradients are bitwise those of the per-step rebuild, except the per-channel gradients that lfi_flowstep_bwd reduces with
    float atomics across CTAs: those vary in the last bits from one identical call to the next, on either path."""
    from lets_face_it_b200 import _cabi as cabi
    from lets_face_it_b200.glow import FlowNet

    np.random.seed(9)
    torch.manual_seed(9)
    C, H, D, Fr, B, K = 12, 16, 24, 40, 21, 3
    net = FlowNet(C, H, D, K, 1, flow_permutation="invconv", flow_coupling="affine", LU_decomposed=True, scale_eps=1e-4,
                  feature_encoder_dim=Fr, glow_rnn_type="gru")
    for l in net.layers:
        l.actnorm.inited = True
    net = net.to(DEV)
    x, c = torch.randn(B, C, device=DEV), torch.randn(B, Fr, device=DEV)
    L = cabi.lib()

    def run(per_step_refresh):
        net.init_rnn_hidden()
        net.zero_grad()
        n0 = L.lfi_launch_count()
        if per_step_refresh:  # what encode did before: every step rebuilt the whole cache
            eng = net._eng()
            eng.ensure(x.device)
            eng.refresh(False)
            z, ld = x, torch.zeros(B, device=DEV)
            for layer in net.layers:
                z, ld = layer(z, c, ld, reverse=False, _refresh=True)
        else:
            z, ld = net(x, c, logdet=torch.zeros(B, device=DEV))
        n = L.lfi_launch_count() - n0
        ((z ** 2).sum() - ld.sum()).backward()
        return n, z.detach().clone(), {name: p.grad.clone() for name, p in net.named_parameters()}

    atomic = ("actnorm.bias", "actnorm.logs", "rnn.bias_hh", "final_linear.bias", "final_linear.logs")
    n_old, z_old, g_old = run(True)
    n_new, z_new, g_new = run(False)
    assert n_new < n_old, (n_new, n_old)
    assert torch.equal(z_new, z_old)
    for name, g in g_new.items():
        if name.endswith(atomic):
            assert relerr(g, g_old[name]) <= 1e-6, name
        else:
            assert torch.equal(g, g_old[name]), name
