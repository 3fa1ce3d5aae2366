"""GPU: FlowStep / FlowNet in the reverse direction under autograd.  In the reference, FlowStep.reverse_flow (models.py:345-373) and
FlowNet.decode (models.py:444-462) are plain torch, so latent optimisation through the decoder and reconstruction losses through
decode get gradients; only Glow.reverse_flow runs under no_grad.  Here every FlowStep.forward(reverse=True) call under autograd is
one node (lfi_flowstep_rev_fwd_train / lfi_flowstep_rev_bwd), checked against the oracle's reverse flow_step / flow_decode
differentiated by torch in CPU fp32: gradients with respect to every latent frame, conditioning vector, the carried state and
every parameter."""
import numpy as np
import pytest
import torch

from oracle import glow_oracle as O
from tests.helpers import relerr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FINAL = dict(C=56, H=128, D=512, F=1560, B=256)


def _hyper(C, K, H, D, rnn, coupling, LU):
    return O.Hyper(C=C, K=K, H=H, D=D, rnn_type=rnn, scale_eps=1e-4, actnorm_scale=1.0, LU=LU, coupling=coupling,
                   hist={m: 1 for m in O.MODALITIES}, enc={m: "none" for m in O.MODALITIES}, enc_hidden={m: 0 for m in O.MODALITIES},
                   in_dim={m: 1 for m in O.MODALITIES}, dropout={m: 0.0 for m in O.MODALITIES})


def _net(rnn, coupling, C, LU=True, K=3, H=16, D=24, Fr=40, seed=3):
    """FlowNet with its ActNorm / LinearZeros / 1x1 weights off their identity-like inits, so that every parameter matters."""
    from lets_face_it_b200.glow import FlowNet

    np.random.seed(seed)
    torch.manual_seed(seed)
    net = FlowNet(C, H, D, K, 1, flow_permutation="invconv", flow_coupling=coupling, LU_decomposed=LU, scale_eps=1e-4,
                  feature_encoder_dim=Fr, glow_rnn_type=rnn)
    gen = torch.Generator().manual_seed(seed + 6)
    with torch.no_grad():
        for n, p in net.named_parameters():
            if "final_linear" in n or "actnorm" in n:
                p.copy_(torch.randn(p.shape, generator=gen) * 0.15)
            elif n.endswith("invconv.weight"):
                p.add_(0.1 * torch.randn(p.shape, generator=gen))
    for l in net.layers:
        l.actnorm.inited = True
    return net


def _worst(pairs):
    return max(relerr(a, b) for a, b in pairs)


# ------------------------------------------------------------------------------------------------ 1. FlowNet.decode per frame
@pytest.mark.parametrize("rnn,coupling,C,LU", [("gru", "affine", 56, True), ("lstm", "affine", 10, True), ("gru", "additive", 7, True),
                                               ("gru", "affine", 12, False)])
def test_flownet_decode_per_frame_gradients(rnn, coupling, C, LU):
    """FlowNet.decode (K = 3) driven frame by frame for three frames with the RNN state carried on the modules, loss =
    sum R x + sum R_l logdet: d loss / d (latents, conditioning, parameters) against torch autograd on the oracle."""
    K, Fr, B, T = 3, 40, 21, 3
    net = _net(rnn, coupling, C, LU)
    hy = _hyper(C, K, 16, 24, rnn, coupling, LU)
    P = O.clone_params({"glow.flow." + k: v for k, v in net.state_dict().items()}, requires_grad=True)
    g = torch.Generator().manual_seed(5)
    zs = [torch.randn(B, C, generator=g).requires_grad_(True) for _ in range(T)]
    conds = [torch.randn(B, Fr, generator=g).requires_grad_(True) for _ in range(T)]
    Rs = [torch.randn(B, C, generator=g) for _ in range(T)]
    Rls = [torch.randn(B, generator=g) for _ in range(T)]
    state, loss_ref, xs_ref = {}, 0.0, []
    for z, c, R, Rl in zip(zs, conds, Rs, Rls):
        x, ld = O.flow_decode(P, hy, z, c, state)
        xs_ref.append(x.detach())
        loss_ref = loss_ref + (x * R).sum() + (ld * Rl).sum()
    loss_ref.backward()

    net = net.to(DEV)
    dz = [z.detach().to(DEV).requires_grad_(True) for z in zs]
    dc = [c.detach().to(DEV).requires_grad_(True) for c in conds]
    net.init_rnn_hidden()
    loss, xs = 0.0, []
    for z, c, R, Rl in zip(dz, dc, Rs, Rls):
        x, ld = net(z, c, reverse=True)
        assert x.requires_grad and ld.requires_grad
        xs.append(x)
        loss = loss + (x * R.to(DEV)).sum() + (ld * Rl.to(DEV)).sum()
    loss.backward()
    e_val = _worst(zip(xs, xs_ref))
    e_in = _worst([(a.grad, b.grad) for a, b in zip(dz + dc, zs + conds)])
    e_par = 0.0
    for n, p in net.named_parameters():
        ref = P["glow.flow." + n].grad
        assert p.grad is not None, n
        e = relerr(p.grad.reshape(ref.shape), ref)
        assert e < 3e-3, (n, e)
        e_par = max(e_par, e)
    print("decode %s/%s C=%d LU=%s: values %.2e, input grads %.2e, parameter grads %.2e" % (rnn, coupling, C, LU, e_val, e_in, e_par))
    assert e_val < 1e-4
    assert e_in < 2e-3


# ------------------------------------------------------------------------------------------------ 2. both inverse kernels, final shapes
def _final_step(rnn, seed=4):
    from lets_face_it_b200.glow import FlowStep

    np.random.seed(seed)
    torch.manual_seed(seed)
    s = FINAL
    step = FlowStep(s["C"], s["H"], s["D"], flow_permutation="invconv", flow_coupling="affine", LU_decomposed=True, scale_eps=1e-4,
                    feature_encoder_dim=s["F"], glow_rnn_type=rnn)
    gen = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for n, p in step.named_parameters():
            if "final_linear" in n or "actnorm" in n:
                p.copy_(torch.randn(p.shape, generator=gen) * 0.15)
    step.actnorm.inited = True
    return step


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return " ".join(e.name for e in prof.events())


@pytest.mark.parametrize("rnn,rows,kernel", [("gru", True, "core_inv_rows"), ("gru", False, "core_inv_persistent"),
                                             ("lstm", True, "core_inv_persistent")])
def test_reverse_step_final_shapes(rnn, rows, kernel, monkeypatch):
    """One reverse step at final_model.yaml shapes (C 56, H 128, D 512, F 1560, B 256) from a carried state: input, conditioning,
    state and parameter gradients against the oracle, through the row-owned inverse kernel (GRU) and the persistent one
    (LFI_INV_ROWS=0, LSTM); the profiler shows which one ran."""
    if not rows:
        monkeypatch.setenv("LFI_INV_ROWS", "0")
    s = FINAL
    B, C, H = s["B"], s["C"], s["H"]
    step = _final_step(rnn)
    hy = _hyper(C, 1, H, s["D"], rnn, "affine", True)
    P = O.clone_params({"glow.flow.layers.0." + k: v for k, v in step.state_dict().items()}, requires_grad=True)
    g = torch.Generator().manual_seed(7)
    x, c = torch.randn(B, C, generator=g), torch.randn(B, s["F"], generator=g)
    h0, c0 = torch.randn(B, H, generator=g) * 0.5, torch.randn(B, H, generator=g) * 0.5
    R, Rl, Rh, Rc = torch.randn(B, C, generator=g), torch.randn(B, generator=g), torch.randn(B, H, generator=g), torch.randn(B, H, generator=g)
    leaves = [t.clone().requires_grad_(True) for t in (x, c, h0, c0)]
    state = {0: leaves[2] if rnn == "gru" else (leaves[2], leaves[3])}
    y, ld = O.flow_step(P, hy, 0, leaves[0], leaves[1], torch.zeros(B), True, state)
    hn, cn = (state[0], None) if rnn == "gru" else state[0]
    loss = (y * R).sum() + (ld * Rl).sum() + (hn * Rh).sum() + ((cn * Rc).sum() if cn is not None else 0.0)
    loss.backward()

    step = step.to(DEV)
    dl = [t.to(DEV).requires_grad_(True) for t in (x, c, h0, c0)]
    out = {}

    def run():
        step.f.hidden, step.f.cell = dl[2], (dl[3] if rnn == "lstm" else None)
        out["y"], out["ld"] = step(dl[0], dl[1], torch.zeros(B, device=DEV), reverse=True)

    assert kernel in _kernel_names(run)
    yd, ldd = out["y"], out["ld"]
    assert relerr(yd, y) < 1e-4 and relerr(ldd, ld) < 1e-4 and relerr(step.f.hidden, hn) < 1e-4
    lossd = (yd * R.to(DEV)).sum() + (ldd * Rl.to(DEV)).sum() + (step.f.hidden * Rh.to(DEV)).sum()
    if rnn == "lstm":
        lossd = lossd + (step.f.cell * Rc.to(DEV)).sum()
    lossd.backward()
    n_in = 4 if rnn == "lstm" else 3
    e_in = _worst([(a.grad, b.grad) for a, b in zip(dl[:n_in], leaves[:n_in])])
    e_par = 0.0
    for n, p in step.named_parameters():
        e = relerr(p.grad, P["glow.flow.layers.0." + n].grad)
        assert e < 3e-3, (n, e)
        e_par = max(e_par, e)
    print("reverse step %s via %s: input/state grads %.2e, parameter grads %.2e" % (rnn, kernel, e_in, e_par))
    assert e_in < 2e-3


# ------------------------------------------------------------------------------------------------ 3. values unchanged
@pytest.mark.parametrize("rnn,rows", [("gru", True), ("gru", False), ("lstm", True)])
def test_reverse_values_do_not_depend_on_grad_mode(rnn, rows, monkeypatch):
    """Under autograd, y / h / c are bitwise those of the no-grad call (the same inverse kernels run) and y requires grad; with
    nothing requiring grad no node is built.  logdet is bitwise equal through core_inv_persistent; core_inv_rows sums a row's
    log-det terms with shared-memory atomics, so there it varies in the last bits between two identical no-grad calls already."""
    from lets_face_it_b200.glow import FlowStep

    if not rows:
        monkeypatch.setenv("LFI_INV_ROWS", "0")
    np.random.seed(4)
    torch.manual_seed(4)
    C, H, D, Fr, B = 56, 128, 64, 80, 33
    step = FlowStep(C, H, D, flow_permutation="invconv", flow_coupling="affine", LU_decomposed=True, scale_eps=1e-4,
                    feature_encoder_dim=Fr, glow_rnn_type=rnn)
    with torch.no_grad():
        for n, p in step.named_parameters():
            if "final_linear" in n or "actnorm" in n:
                p.normal_(0, 0.15)
    step.actnorm.inited = True
    step = step.to(DEV)
    x, c = torch.randn(B, C, device=DEV), torch.randn(B, Fr, device=DEV)
    h0, c0 = torch.randn(B, H, device=DEV), (torch.randn(B, H, device=DEV) if rnn == "lstm" else None)

    def call(logdet):
        step.f.hidden, step.f.cell = h0, c0
        y, ld = step(x, c, logdet, reverse=True)
        return y, ld, step.f.hidden, step.f.cell

    for logdet in (torch.linspace(-1, 1, B, device=DEV), 0.0, None):
        with torch.no_grad():
            ref = call(logdet)
        got = call(logdet)
        assert got[0].requires_grad and got[2].requires_grad
        for i, (a, b) in enumerate(zip(got, ref)):
            if i == 1 and a is not None and rnn == "gru" and rows:
                assert relerr(a, b) <= 1e-6
            else:
                assert (a is None and b is None) or torch.equal(a, b)
    for p in step.parameters():
        p.requires_grad_(False)
    y, ld, h, _ = call(0.0)
    assert y.grad_fn is None and ld.grad_fn is None and h.grad_fn is None


# ------------------------------------------------------------------------------------------------ 4. round trip
@pytest.mark.parametrize("rnn", ["gru", "lstm"])
def test_decode_encode_round_trip_gradient(rnn):
    """decode(encode(x)) from the same initial state is the identity, so d/dx sum R decode(encode(x)) = R."""
    C, Fr, B, H = 12, 40, 21, 16
    net = _net(rnn, "affine", C).to(DEV)
    g = torch.Generator().manual_seed(11)
    x = torch.randn(B, C, generator=g).to(DEV).requires_grad_(True)
    c = torch.randn(B, Fr, generator=g).to(DEV)
    R = torch.randn(B, C, generator=g).to(DEV)
    h0 = [torch.randn(B, H, generator=g).to(DEV) * 0.5 for _ in net.layers]
    c0 = [torch.randn(B, H, generator=g).to(DEV) * 0.5 if rnn == "lstm" else None for _ in net.layers]

    def set_state():
        for l, h, cc in zip(net.layers, h0, c0):
            l.f.hidden, l.f.cell = h, cc

    set_state()
    z, _ = net(x, c, logdet=torch.zeros(B, device=DEV))
    set_state()
    xr, _ = net(z, c, reverse=True)
    assert relerr(xr, x) < 1e-4
    (xr * R).sum().backward()
    err = float((x.grad - R).abs().max() / R.abs().max())
    print("round trip %s: |dx - R| / max|R| = %.2e" % (rnn, err))
    assert err <= 1e-4


# ------------------------------------------------------------------------------------------------ 5. determinism
@pytest.mark.parametrize("rnn", ["gru", "lstm"])
def test_reverse_backward_is_bitwise_deterministic(rnn):
    """Two identical backward calls give bitwise-equal gradients for every input and parameter (fixed-order reductions, no float
    atomics, no split-K); B is large enough that the row reductions are long."""
    C, Fr, B = 56, 80, 2048
    net = _net(rnn, "affine", C, H=128, D=64, Fr=Fr).to(DEV)
    g = torch.Generator().manual_seed(12)
    zs = [torch.randn(B, C, generator=g).to(DEV) for _ in range(2)]
    cs = [torch.randn(B, Fr, generator=g).to(DEV) for _ in range(2)]
    R = torch.randn(B, C, generator=g).to(DEV)
    grads = []
    for _ in range(2):
        net.init_rnn_hidden()
        net.zero_grad()
        dz = [z.clone().requires_grad_(True) for z in zs]
        dc = [c.clone().requires_grad_(True) for c in cs]
        loss = 0.0
        for z, c in zip(dz, dc):
            x, ld = net(z, c, reverse=True)
            loss = loss + (x * R).sum() + ld.sum()
        loss.backward()
        grads.append([t.grad.clone() for t in dz + dc] + [p.grad.clone() for p in net.parameters()])
    assert all(torch.equal(a, b) for a, b in zip(*grads))


# ------------------------------------------------------------------------------------------------ 6. one refresh per decode
def test_flownet_decode_refreshes_once_under_autograd():
    """FlowNet.decode under autograd rebuilds the derived weight cache (with W^-1) once per call, not once per step, with bitwise
    equal outputs and gradients."""
    from lets_face_it_b200 import _cabi as cabi

    C, Fr, B = 12, 40, 21
    net = _net("gru", "affine", C).to(DEV)
    net._eng().ensure(torch.device(DEV))  # the FlowNet's engine, before any step builds one of its own
    g = torch.Generator().manual_seed(13)
    z0, c = torch.randn(B, C, generator=g).to(DEV), torch.randn(B, Fr, generator=g).to(DEV)
    L = cabi.lib()

    def run(per_step_refresh):
        net.init_rnn_hidden()
        net.zero_grad()
        z = z0.clone().requires_grad_(True)
        n0 = L.lfi_launch_count()
        if per_step_refresh:
            x, ld = z, 0.0
            for layer in reversed(net.layers):
                x, ld = layer(x, c, ld, reverse=True, _refresh=True)
        else:
            x, ld = net(z, c, reverse=True)
        n = L.lfi_launch_count() - n0
        ((x ** 2).sum() - ld.sum()).backward()
        return n, x.detach().clone(), [z.grad.clone()] + [p.grad.clone() for p in net.parameters()]

    n_old, x_old, g_old = run(True)
    n_new, x_new, g_new = run(False)
    assert n_new < n_old, (n_new, n_old)
    assert torch.equal(x_new, x_old)
    assert all(torch.equal(a, b) for a, b in zip(g_new, g_old))
