"""The fused trainer with SGD and RMSprop, and its state: the clip + SGD / RMSprop kernels against torch.optim, `Trainer` against
the drop-in's autograd path driven by torch.optim, checkpoint / resume, `GraphedStep`, and the exchange of optimizer state with
torch.optim (configure_optimizers of lets_face_it_glow.py:61-72)."""
import copy
import functools
import io

import pytest
import torch

from tests.helpers import final_hparams, relerr, small_hparams
from tests.kat import build_kat_model, kat_batch, to_device

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0) if torch.cuda.is_available() else None

SGD_CASES = [dict(momentum=0.0), dict(momentum=0.9), dict(momentum=0.9, dampening=0.1), dict(momentum=0.9, nesterov=True),
             dict(momentum=0.0, weight_decay=1e-2), dict(momentum=0.9, weight_decay=1e-2, nesterov=True)]
# Centered with weight decay: at n_theta the clipped gradients are ~5e-3 per element, and a decay term that dominates them makes
# g the same from step to step, so sq - grad_avg^2 cancels to rounding level and its last bits decide avg (in torch as here):
# the decay stays below the gradients in that case.
RMS_CASES = [dict(), dict(centered=True), dict(momentum=0.9), dict(weight_decay=1e-2),
             dict(alpha=0.9, centered=True, momentum=0.9, weight_decay=1e-4)]
# the configuration of each optimizer that the trainer-level tests run
TRAIN_CASES = [("adam", {"betas": (0.9, 0.9999), "eps": 1e-8}), ("sgd", {"momentum": 0.9, "nesterov": True}),
               ("rmsprop", {"centered": True, "momentum": 0.9})]
LR = {"adam": 1e-3, "sgd": 1e-2, "rmsprop": 1e-3}


@functools.lru_cache(None)
def _n_theta():
    return build_kat_model(final_hparams(), DEV).engine().n_theta


def _fused(name, args, theta, g, bufs, n, hyper, max_norm, gscale, scratch):
    from lets_face_it_b200 import _cabi as cabi

    L, p = cabi.lib(), lambda k: bufs[k].data_ptr() if k in bufs else None
    if name == "sgd":
        cabi.check(L.lfi_clip_sgd_dev(theta.data_ptr(), g.data_ptr(), p("momentum_buffer"), n, hyper.data_ptr(), args.get("momentum", 0.0),
                                      args.get("dampening", 0.0), args.get("weight_decay", 0.0), int(args.get("nesterov", False)), max_norm,
                                      gscale, scratch.data_ptr(), cabi.stream_ptr()), "lfi_clip_sgd_dev")
    else:
        cabi.check(L.lfi_clip_rmsprop_dev(theta.data_ptr(), g.data_ptr(), p("square_avg"), p("grad_avg"), p("momentum_buffer"), n,
                                          hyper.data_ptr(), args.get("alpha", 0.99), args.get("eps", 1e-8), args.get("weight_decay", 0.0),
                                          args.get("momentum", 0.0), max_norm, gscale, scratch.data_ptr(), cabi.stream_ptr()),
                   "lfi_clip_rmsprop_dev")


def _run_kernel(name, args, n, max_norm, gscale, steps=4, seed=3):
    """`steps` fused updates and the same steps of clip_grad_norm_ + torch.optim on a copy; returns both states."""
    from lets_face_it_b200.train import _buffer_names, optimizer_args

    gen = torch.Generator(device=DEV).manual_seed(seed)
    theta = torch.randn(n, device=DEV, generator=gen)
    ref = theta.clone().requires_grad_(True)
    lr = 1e-2 if name == "sgd" else 1e-3
    opt = (torch.optim.SGD if name == "sgd" else torch.optim.RMSprop)([ref], lr=lr, **args)
    full = optimizer_args(name, lr, args)
    bufs = {k: torch.zeros(n, device=DEV) for k in _buffer_names(name, full)}
    scratch = torch.zeros(2, device=DEV)
    for st in range(steps):
        g = torch.randn(n, device=DEV, generator=gen) * 3.0
        hyper = torch.tensor([lr, 1.0 if st == 0 else 0.0] if name == "sgd" else [lr], device=DEV)
        _fused(name, args, theta, g, bufs, n, hyper, max_norm, gscale, scratch)
        ref.grad = g * gscale  # what the all-reduce mean hands to the clip: grad_scale = 1 / world
        # clip_grad_norm_ = the norm, then clip_grads_with_norm_.  The norm pass sums in another order than torch (checked here);
        # the reference clips with its result, since RMSprop's first steps are ~ lr * sign(g) and weight decay makes g cancel to
        # rounding level for some elements, whose sign then follows the last bit of the clip coefficient.
        norm = torch.sqrt(scratch[0]) * gscale
        assert abs(float(norm) / float(ref.grad.double().norm()) - 1) < 1e-5
        if max_norm > 0:
            torch.nn.utils.clip_grads_with_norm_([ref], max_norm, norm)
        opt.step()
    return theta, bufs, ref.detach(), opt.state[ref]


@pytest.mark.parametrize("name,args", [("sgd", a) for a in SGD_CASES] + [("rmsprop", a) for a in RMS_CASES])
def test_clip_update_matches_torch(name, args):
    """θ and every buffer after 4 steps of the clip + torch.optim at n = 100,003 (ragged tail) and n = n_theta of final_model.yaml,
    gradients of scale 3 (the clip at 20 engages) and no clip, grad_scale 1 and 0.5, within the bound of
    test_clip_adam_matches_torch."""
    for n in (100003, _n_theta()):
        for max_norm in (20.0, 0.0):
            for gscale in (1.0, 0.5):
                theta, bufs, ref, st = _run_kernel(name, args, n, max_norm, gscale)
                where = (n, max_norm, gscale)
                assert relerr(theta, ref) < 2e-6, where
                for k, b in bufs.items():
                    assert relerr(b, st[k]) < 2e-6, (k,) + where
                assert set(bufs) == {k for k in st if k != "step"}


@pytest.mark.parametrize("name,args", [("sgd", SGD_CASES[5]), ("rmsprop", RMS_CASES[4])])
def test_clip_update_is_bitwise_reproducible(name, args):
    """The update has no atomics: the same state and gradients give bitwise equal θ and buffers.  (No clip here: the norm pass
    sums its blocks with atomics, so the clip coefficient may differ in its last bit from run to run.)"""
    a = _run_kernel(name, args, 100003, 0.0, 1.0)
    b = _run_kernel(name, args, 100003, 0.0, 1.0)
    assert torch.equal(a[0], b[0])
    for k in a[1]:
        assert torch.equal(a[1][k], b[1][k]), k


# ------------------------------------------------------------------------------------------------ Trainer
def _hp(case, name, args):
    hp = copy.deepcopy(small_hparams("gru") if case == "small" else final_hparams())
    hp.Optim = {"name": name, "args": {name: dict(args)}, "Schedule": hp.Optim.get("Schedule")}
    return hp


def _model(hp, mode, ddi_batch):
    """The KAT model after the ActNorm data-dependent init on `ddi_batch` (run here, so that both sides of a comparison start
    from it; `inited` is not part of a state dict, as in the reference)."""
    from lets_face_it_b200 import _cabi as cabi

    m = build_kat_model(hp, DEV).train()
    m.gemm_mode = {"fp32": cabi.GEMM_FP32, "bf16x3": cabi.GEMM_BF16X3}[mode]
    m._ddi(m.engine(), ddi_batch, None)
    return m


def _batches(hp, case, n, seed=60):
    B, T = (6, 30) if case == "small" else (32, 40)
    return [to_device(kat_batch(hp, B, T, seed=seed + i), DEV) for i in range(n)]


def _torch_step(m, opt, batch, max_norm):
    opt.zero_grad()
    _, loss, _ = m(batch)
    loss.backward()
    torch.nn.utils.clip_grad_norm_(m.parameters(), max_norm)
    opt.step()
    return float(loss)


def _params(m):
    return {n: p.detach().clone() for n, p in m.named_parameters()}


def _check_delta(d_got, d_ref):
    """θ_after − θ_before per tensor, with the bounds of test_three_optimizer_steps_against_reference."""
    worst = ("", 0.0)
    for n in d_ref:
        ref, got = d_ref[n].double(), d_got[n].double()
        assert abs(float(got.norm()) - float(ref.norm())) < 0.02 * float(ref.norm()) + 1e-12, n
        err = float((got - ref).norm() / ref.norm().clamp_min(1e-30))
        worst = max(worst, (n, err), key=lambda t: t[1])
    assert worst[1] < 0.05, worst


@pytest.mark.parametrize("case,mode", [("small", "fp32"), ("full", "bf16x3")])
@pytest.mark.parametrize("name,args", TRAIN_CASES[1:])
def test_trainer_matches_torch_optim_on_autograd_path(case, mode, name, args):
    """3 Trainer.steps against 3 steps of SeqGlow.forward -> backward -> clip_grad_norm_ -> torch.optim on a second copy."""
    from lets_face_it_b200.train import OPTIMIZERS, Trainer

    hp = _hp(case, name, args)
    batches = _batches(hp, case, 3)
    m = _model(hp, mode, batches[0])
    tr = Trainer(m, dropout=False, lr=LR[name])
    m2 = _model(hp, mode, batches[0])
    opt = OPTIMIZERS[name](m2.parameters(), lr=LR[name], **args)
    t1, t2 = _params(m), _params(m2)
    for b in batches:
        lf, lt = float(tr.step(b)), _torch_step(m2, opt, b, tr.max_norm)
        assert abs(lf - lt) < 2e-5 * abs(lt), (lf, lt)
    p1, p2 = _params(m), _params(m2)
    _check_delta({n: p1[n] - t1[n] for n in t1}, {n: p2[n] - t2[n] for n in t2})


@pytest.mark.parametrize("name,args", TRAIN_CASES)
def test_trainer_launches_the_chosen_update(name, args):
    """Optim.name decides the kernel: Adam's step still runs clip_adam_kernel (and nothing else of the optimizers)."""
    from torch.profiler import ProfilerActivity, profile

    from lets_face_it_b200.train import Trainer

    hp = _hp("small", name, args)
    b = _batches(hp, "small", 1)[0]
    tr = Trainer(_model(hp, "fp32", b), dropout=False)
    tr.step(b)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        tr.step(b)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    kernels = {k: sum(k in n for n in names) for k in ("clip_adam_kernel", "clip_sgd_kernel", "clip_rmsprop_kernel", "sumsq_kernel")}
    assert kernels == {"clip_adam_kernel": int(name == "adam"), "clip_sgd_kernel": int(name == "sgd"),
                       "clip_rmsprop_kernel": int(name == "rmsprop"), "sumsq_kernel": 1}, kernels


# ------------------------------------------------------------------------------------------------ checkpoint / resume
def _run_to_run(pa, pb):
    """The bound of test_graphed_steps_equal_eager_steps: per tensor |a - b| / |a| < 1e-3.  Returns the worst tensor."""
    return max(((n, float((pa[n] - pb[n]).double().norm() / pa[n].double().norm().clamp_min(1e-12))) for n in pa), key=lambda t: t[1])


@pytest.mark.parametrize("name,args", TRAIN_CASES)
def test_resume_continues_the_run(name, args):
    """Run A: 5 steps.  Run B: 2 steps, torch.save / torch.load of model and trainer state, a fresh model and Trainer, 3 more
    steps on the same batches.  A restart from the model state alone must not continue the run."""
    from lets_face_it_b200.train import Trainer

    hp = _hp("small", name, args)
    batches = _batches(hp, "small", 5)

    def run(steps, tr=None):
        tr = tr or Trainer(_model(hp, "fp32", batches[0]), dropout=False, lr=LR[name])
        losses = [float(tr.step(b)) for b in steps]
        return tr, losses

    tra, la = run(batches[:2])
    a2 = _params(tra.model)
    _, la5 = run(batches[2:], tra)
    a5 = _params(tra.model)

    trb, _ = run(batches[:2])
    b2 = _params(trb.model)
    sd = trb.state_dict()
    assert sd["step_count"] == 2
    buf = io.BytesIO()
    torch.save({"model": trb.model.state_dict(), "trainer": sd}, buf)
    trb.step(batches[2])  # the saved dict is a snapshot
    assert sd["step_count"] == 2 and all(not torch.equal(v, trb.buffers[k]) for k, v in sd["buffers"].items())
    buf.seek(0)
    ck = torch.load(buf)
    results = {}
    for load_trainer in (True, False):
        m = _model(hp, "fp32", batches[0])
        m.load_state_dict(ck["model"])
        tr = Trainer(m, dropout=False, lr=LR[name])
        if load_trainer:
            tr.load_state_dict(ck["trainer"])
            assert tr.step_count == 2
        _, losses = run(batches[2:], tr)
        p5 = _params(m)
        results[load_trainer] = (losses, {n: p5[n] - b2[n] for n in p5})
    losses, d = results[True]
    for x, y in zip(losses, la5):
        assert abs(x - y) < 2e-5 * abs(y), (losses, la5)
    # θ5 − θ2 of run B added to run A's θ2: within the run-to-run bound of run A's θ5 (fails without the trainer state)
    assert _run_to_run(a5, {n: a2[n] + d[n] for n in d})[1] < 1e-3
    assert _run_to_run(a5, {n: a2[n] + results[False][1][n] for n in d})[1] > 1e-3


@pytest.mark.parametrize("name,args", TRAIN_CASES)
def test_load_state_dict_of_state_dict_is_the_identity(name, args):
    from lets_face_it_b200.train import Trainer

    hp = _hp("small", name, args)
    batches = _batches(hp, "small", 2)
    tr = Trainer(_model(hp, "fp32", batches[0]), dropout=False, lr=LR[name])
    for b in batches:
        tr.step(b)
    sd = tr.state_dict()
    tr.load_state_dict(sd)
    sd2 = tr.state_dict()
    assert set(sd) == set(sd2)
    for k in sd:
        if k == "buffers":
            assert all(torch.equal(sd[k][j], sd2[k][j]) for j in sd[k])
        else:
            assert sd[k] == sd2[k], k
    other = "sgd" if name != "sgd" else "adam"
    with pytest.raises(ValueError, match="%s.*%s" % (other, name)):
        tr.load_state_dict({**sd, "optimizer": other})


@pytest.mark.parametrize("name,args", TRAIN_CASES[1:])
def test_graphed_steps_equal_eager_steps_and_follow_loads(name, args):
    """As test_graphed_steps_equal_eager_steps for Adam: 2 eager steps + 4 replays against 6 eager steps.  Then loads into the
    trainer that holds the graph: the state of the eager run after step 3 (replays of batches 3..5 must give that run's steps 4..6),
    and a state saved before any step (SGD: the buffer is empty again, so the next replay is a first momentum step)."""
    from lets_face_it_b200.train import Trainer

    hp = _hp("small", name, args)
    batches = _batches(hp, "small", 6)
    me = _model(hp, "fp32", batches[0])
    tre = Trainer(me, dropout=False, lr=LR[name])
    snaps, le = [], []
    for b in batches:
        snaps.append((copy.deepcopy(me.state_dict()), tre.state_dict()))
        le.append(float(tre.step(b)))
    pe = _params(me)

    mg = _model(hp, "fp32", batches[0])
    trg = Trainer(mg, dropout=False, lr=LR[name])
    lg = [float(trg.step(batches[0]))]
    gs = trg.graphed(batches[1], warmup=1)
    lg.append(None)
    lg += [float(gs.step(b)) for b in batches[2:]]
    assert trg.step_count == 6
    for st in (0, 2, 3, 4, 5):
        assert abs(le[st] - lg[st]) < 2e-5 * abs(le[st]) + 1e-6, (st, le[st], lg[st])
    assert abs(le[5] - le[0]) > 1e-3 * abs(le[0])
    assert _run_to_run(pe, _params(mg))[1] < 1e-3

    for start in (0, 3):
        mg.load_state_dict(snaps[start][0])
        trg.load_state_dict(snaps[start][1])
        got = [float(gs.step(b)) for b in batches[start:start + 3]]
        for st, x in zip(range(start, start + 3), got):
            assert abs(le[st] - x) < 2e-5 * abs(le[st]) + 1e-6, (start, st, le[st], x)
    assert _run_to_run(pe, _params(mg))[1] < 1e-3  # after the load of step 3's state: the eager run's end


# ------------------------------------------------------------------------------------------------ exchange with torch.optim
def _same_format(got, want):
    assert got["param_groups"] == want["param_groups"]
    assert set(got["state"]) == set(want["state"])
    for i, st in want["state"].items():
        assert set(got["state"][i]) == set(st), i
        for k, v in st.items():
            g = got["state"][i][k]
            assert (g.dtype, g.shape, g.device) == (v.dtype, v.shape, v.device), (i, k)


@pytest.mark.parametrize("name,args", TRAIN_CASES + [("sgd", {"momentum": 0.0, "weight_decay": 1e-3})])
def test_exchange_with_torch_optim(name, args):
    """torch -> fused: 2 autograd steps with torch.optim, its state_dict() into a fresh Trainer, 1 step on each side.
    fused -> torch: 2 Trainer steps, optimizer_state_dict() into a fresh torch.optim, 1 step on each side.  The exported
    dict has the format of the real optimizer's after the same steps."""
    from lets_face_it_b200.train import OPTIMIZERS, Trainer

    hp = _hp("small", name, args)
    b = _batches(hp, "small", 3)
    lr = LR[name]

    # torch -> fused
    mt = _model(hp, "fp32", b[0])
    opt = OPTIMIZERS[name](mt.parameters(), lr=lr, **args)
    for x in b[:2]:
        _torch_step(mt, opt, x, 20.0)
    mf = _model(hp, "fp32", b[0])
    mf.load_state_dict(mt.state_dict())
    tr = Trainer(mf, dropout=False, lr=0.5)  # the lr comes from the loaded dict
    tr.load_optimizer_state_dict(opt.state_dict())
    assert tr.lr == lr
    if name != "sgd":
        assert tr.step_count == 2
    t2 = _params(mt)
    lf, lt = float(tr.step(b[2])), _torch_step(mt, opt, b[2], 20.0)
    assert abs(lf - lt) < 2e-5 * abs(lt)
    if name == "adam":
        assert tr.step_count == 3
    pf, pt = _params(mf), _params(mt)
    _check_delta({n: pf[n] - t2[n] for n in t2}, {n: pt[n] - t2[n] for n in t2})
    _same_format(tr.optimizer_state_dict(), opt.state_dict())

    # fused -> torch
    mf = _model(hp, "fp32", b[0])
    tr = Trainer(mf, dropout=False, lr=lr)
    for x in b[:2]:
        tr.step(x)
    mt = _model(hp, "fp32", b[0])
    mt.load_state_dict(mf.state_dict())
    opt = OPTIMIZERS[name](mt.parameters(), lr=0.5, **args)
    opt.load_state_dict(tr.optimizer_state_dict())
    assert opt.param_groups[0]["lr"] == lr
    t2 = _params(mf)
    lf, lt = float(tr.step(b[2])), _torch_step(mt, opt, b[2], 20.0)
    assert abs(lf - lt) < 2e-5 * abs(lt)
    pf, pt = _params(mf), _params(mt)
    _check_delta({n: pf[n] - t2[n] for n in t2}, {n: pt[n] - t2[n] for n in t2})


def test_exchange_rejects_foreign_or_partial_state():
    from lets_face_it_b200.train import Trainer

    hp = _hp("small", "adam", TRAIN_CASES[0][1])
    b = _batches(hp, "small", 1)[0]
    m = _model(hp, "fp32", b)
    tr = Trainer(m, dropout=False)
    sgd = torch.optim.SGD(m.parameters(), lr=0.1, momentum=0.9)
    with pytest.raises(ValueError, match="Adam"):
        tr.load_optimizer_state_dict(sgd.state_dict())
    tr.step(b)
    sd = tr.optimizer_state_dict()
    del sd["state"][3]
    with pytest.raises(ValueError, match="parameter 3"):
        tr.load_optimizer_state_dict(sd)
    sd = tr.optimizer_state_dict()
    sd["state"][0]["step"] = torch.tensor(7.0)
    with pytest.raises(ValueError, match="step"):
        tr.load_optimizer_state_dict(sd)
