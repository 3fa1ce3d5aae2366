"""TEST INFRASTRUCTURE ONLY — generates `tests/golden/*.npz` by running the UNMODIFIED reference
(`code/glow_pytorch/glow` of a jonepatr/lets_face_it checkout) on the CPU.

    LFI_REFERENCE_ROOT=<checkout> python oracle/make_golden.py    # writes tests/golden/kat_full.npz, kat_small_*.npz

Recipe = SURVEY.md §8(c): torch/numpy seed 1234 (code/config.toml:4), LinearZeros perturbed from
Generator(7), encoder dropout disabled (or replaced by injected masks), data from Generator(1),
one training-mode pass for ActNorm data-dependent init, then eval-mode forward / inference /
invert and a training-mode backward.  The reference cannot travel to the GPU box, so the vectors
are committed together with this script.
"""
import argparse
import copy
import os
import sys

import numpy as np
import torch
import torch.nn as nn

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import glow_oracle as O  # noqa: E402
from oracle.ref_shim import import_reference, load_reference_hparams  # noqa: E402
from tests.kat import fingerprint  # noqa: E402  (the stored fingerprints and the test must sum alike)

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def small_hparams(rnn_type="gru"):
    hp = load_reference_hparams()
    hp = copy.deepcopy(hp)
    hp.Conditioning["cond_dim"] = 24
    hp.Conditioning["p1_face"]["dim"] = 12
    hp.Conditioning["p2_face"]["dim"] = 12
    hp.Conditioning["p1_face"]["history"] = 3
    hp.Conditioning["p2_face"]["history"] = 6
    hp.Conditioning["p2_face"]["hidden_dim"] = 8
    hp.Conditioning["p1_speech"]["history"] = 2
    hp.Conditioning["p1_speech"]["hidden_dim"] = 6
    hp.Conditioning["p2_speech"]["history"] = 4
    hp.Conditioning["p2_speech"]["hidden_dim"] = 8
    hp.Data["speech_dim"] = 5
    hp.Glow["K"] = 3
    hp.Glow["hidden_channels"] = 16
    hp.Glow["rnn_type"] = rnn_type
    hp.Validation["scale_logging"] = False
    return hp


class _LSTMZero(nn.LSTMCell):
    """`(None, None)` -> zero state: the evident intent of models.py:209-213 (SURVEY.md §0.1)."""

    def forward(self, x, hx=None):
        if hx is not None and hx[0] is None:
            hx = None
        return super().forward(x, hx)


class _MaskFeeder(nn.Module):
    """Stands in for `nn.Dropout` inside ModalityEncoder (models.py:56-58): returns injected masks."""

    def __init__(self, masks):
        super().__init__()
        self.masks, self.i = masks, 0

    def reset(self):
        self.i = 0

    def forward(self, ones):
        m = self.masks[self.i]
        self.i += 1
        assert m.shape == ones.shape
        return m


def build_reference_model(hp, models, modules):
    torch.manual_seed(1234)
    np.random.seed(1234)
    m = models.SeqGlow(hp)
    g = torch.Generator().manual_seed(7)
    for mod in m.modules():
        if isinstance(mod, modules.LinearZeros):
            with torch.no_grad():
                mod.weight.copy_(torch.randn(mod.weight.shape, generator=g) * 0.05)
                mod.bias.copy_(torch.randn(mod.bias.shape, generator=g) * 0.05)
                mod.logs.copy_(torch.randn(mod.logs.shape, generator=g) * 0.1)
    if hp.Glow["rnn_type"] == "lstm":
        for layer in m.glow.flow.layers:
            layer.f.rnn.__class__ = _LSTMZero
    for mod in m.modules():
        if isinstance(mod, models.ModalityEncoder):
            mod.dropout = None
    return m


def run_case(hp, B, T, infer_len, with_masks, full_tensors, tag):
    models, modules = import_reference()
    hy = O.Hyper.from_hparams(hp)
    m = build_reference_model(hp, models, modules)
    batch = O.synthetic_batch(hy, B, T, seed=1)
    out = {}
    sd_init = {k: v.clone() for k, v in m.state_dict().items()}

    m.train()
    _, loss_ddi, _ = m(batch)  # ActNorm data-dependent init (modules.py:69-70)
    out["loss_ddi"] = loss_ddi.detach().numpy()
    sd = {k: v.clone() for k, v in m.state_dict().items()}

    m.eval()
    z_seq, loss, losses = m(batch)
    z = torch.stack(z_seq)
    nll = torch.stack(losses)
    out["loss"] = loss.detach().numpy()
    out["nll"] = nll.numpy()
    out["z_sum"] = np.float64(z.double().sum())
    out["z_absmean"] = np.float64(z.double().abs().mean())

    # sampling at eps=0 from a zero seed (deterministic), and with injected noise
    hp.Infer["eps"] = 0
    seed_faces = torch.zeros(B, hy.start_ts, hy.C)
    data = dict(batch)
    data["p1_face"] = seed_faces
    x0 = m.inference(infer_len, data=data)
    gn = torch.Generator().manual_seed(11)
    noise = torch.randn(infer_len - hy.start_ts, B, hy.C, generator=gn) * 0.7
    it = iter(noise)
    orig = modules.GaussianDiag.sample
    modules.GaussianDiag.sample = staticmethod(lambda shape, eps_std=1: next(it))
    try:
        hp.Infer["eps"] = 0.7
        x1 = m.inference(infer_len, data=data)
    finally:
        modules.GaussianDiag.sample = orig
    rec, inv_loss = m.invert(z_seq, batch)
    rec = torch.stack(rec)
    out["invert_maxerr"] = np.float64((rec - batch["p1_face"][:, hy.start_ts :].transpose(0, 1)).abs().max())
    out["invert_loss"] = inv_loss.detach().numpy()

    # training-mode backward (dropout disabled)
    m.train()
    m.zero_grad()
    loss_t = m(batch)[1]
    loss_t.backward()
    gnames = [n for n, p in m.named_parameters()]
    gnorms = np.array([float(p.grad.double().norm()) for n, p in m.named_parameters()])
    out["grad_names"] = np.array(gnames)
    out["grad_norms"] = gnorms
    out["grad_total_norm"] = np.float64(np.sqrt((gnorms ** 2).sum()))
    out["loss_train"] = loss_t.detach().numpy()
    grads = {n: p.grad.clone() for n, p in m.named_parameters()}

    if with_masks:
        Tp = T - hy.start_ts
        masks = O.make_masks(hy, B, Tp, seed=3)
        feeders = {}
        for mod_name in O.MODALITIES:
            enc = getattr(m.feature_encoder, mod_name + "_encoder", None)
            if enc is not None and masks[mod_name] is not None:
                feeders[mod_name] = _MaskFeeder(masks[mod_name])
                enc.dropout = feeders[mod_name]
        m.zero_grad()
        z_seq_m, loss_m, losses_m = m(batch)
        loss_m.backward()
        out["masked_loss"] = loss_m.detach().numpy()
        out["masked_nll"] = torch.stack(losses_m).numpy()
        out["masked_grad_norms"] = np.array([float(p.grad.double().norm()) for n, p in m.named_parameters()])
        if full_tensors:
            out["masked_z"] = torch.stack(z_seq_m).numpy()
            for n, p in m.named_parameters():
                out["masked_grad/" + n] = p.grad.numpy().copy()
        else:
            out["masked_z_head"] = torch.stack(z_seq_m)[:, :min(B, 8)].numpy()
            out["masked_z_sum"] = np.float64(torch.stack(z_seq_m).double().sum())
        out["masked_grad_total_norm"] = np.float64(np.sqrt((out["masked_grad_norms"] ** 2).sum()))
        for mod_name, fd in feeders.items():  # back to "dropout disabled" for whatever follows
            getattr(m.feature_encoder, mod_name + "_encoder").dropout = None

    names, fp = fingerprint(sd)
    out["fp_names"] = np.array(names)
    out["fp"] = fp
    names0, fp0 = fingerprint(sd_init)
    out["fp_init"] = fp0
    out["B"], out["T"], out["infer_len"] = B, T, infer_len
    if full_tensors:
        for k, v in sd.items():
            out["param/" + k] = v.numpy()
        for k, v in batch.items():
            out["batch/" + k] = v.numpy()
        out["z"] = z.numpy()
        out["x_eps0"] = x0.numpy()
        out["x_noise"] = x1.numpy()
        out["noise"] = noise.numpy()
        out["rec"] = rec.numpy()
        for n, g_ in grads.items():
            out["grad/" + n] = g_.numpy()
    else:
        nb = min(B, 8)
        out["z_head"] = z[:, :nb].numpy()
        out["x_eps0_head"] = x0[:nb].numpy()
        out["x_noise_head"] = x1[:nb].numpy()
        out["x_eps0_sum"] = np.float64(x0.double().sum())
        out["x_eps0_absmean"] = np.float64(x0.double().abs().mean())
        out["x_noise_sum"] = np.float64(x1.double().sum())
        # the ActNorm parameters after DDI are data dependent: ship them (16*2*56 floats)
        for k, v in sd.items():
            if ".actnorm." in k:
                out["param/" + k] = v.numpy()
    path = os.path.join(GOLDEN, tag + ".npz")
    np.savez_compressed(path, **out)
    print(tag, "loss", float(loss), "grad_norm", float(out["grad_total_norm"]), "->", path,
          "%.1f KB" % (os.path.getsize(path) / 1024))


def run_long_sampling(hp, B, gen_frames, keep, tag):
    """BASELINE.json configs[3] horizon: `SeqGlow.inference` (models.py:567-596) of 30 s = 750 frames at temperature 0.7 with
    injected noise (Generator(21), so the GPU test regenerates it), zero seed frames, KAT model after the DDI pass of the
    B=64 KAT batch.  Stores the first `keep` sequences (sequences are independent)."""
    models, modules = import_reference()
    hy = O.Hyper.from_hparams(hp)
    m = build_reference_model(hp, models, modules)
    m.train()
    m(O.synthetic_batch(hy, 64, 80, seed=1))  # the DDI pass of kat_full
    m.eval()
    seq_len = hy.start_ts + gen_frames
    data = O.synthetic_batch(hy, B, seq_len, seed=5)
    data["p1_face"] = torch.zeros(B, hy.start_ts, hy.C)
    noise = torch.randn(gen_frames, B, hy.C, generator=torch.Generator().manual_seed(21)) * 0.7
    it = iter(noise)
    orig = modules.GaussianDiag.sample
    modules.GaussianDiag.sample = staticmethod(lambda shape, eps_std=1: next(it))
    try:
        hp.Infer["eps"] = 0.7
        x = m.inference(seq_len, data=data)
    finally:
        modules.GaussianDiag.sample = orig
    out = {"B": B, "gen_frames": gen_frames, "x_head": x[:keep].numpy(), "x_sum": np.float64(x.double().sum()),
           "x_absmax_per_frame": x.abs().amax(dim=(0, 2)).numpy()}
    for k, v in m.state_dict().items():
        if ".actnorm." in k:
            out["param/" + k] = v.numpy()
    path = os.path.join(GOLDEN, tag + ".npz")
    np.savez_compressed(path, **out)
    print(tag, "max|x|", float(x.abs().max()), "->", path, "%.1f KB" % (os.path.getsize(path) / 1024))


def run_train_steps(hp, B, T, steps, with_masks, full_tensors, tag):
    """`steps` optimizer steps of the reference's training loop on the live reference: `LetsFaceItGlow.training_step` is
    `loss = seq_glow(batch)[1]` (lets_face_it_glow.py:52), Lightning then runs backward, `clip_grad_norm_(gradient_clip_val)`
    (final_model.yaml:126) and `configure_optimizers`' Adam(lr, betas, eps) (lets_face_it_glow.py:61-72, final_model.yaml:91-95,
    130).  The first step includes the ActNorm DDI (model fresh, training mode).  Stores the loss of every step, the global
    gradient norm before clipping, and theta_after - theta_before per tensor (full tensors for the small case, fingerprints
    plus a few whole tensors for final_model.yaml)."""
    models, modules = import_reference()
    hy = O.Hyper.from_hparams(hp)
    m = build_reference_model(hp, models, modules)
    batch = O.synthetic_batch(hy, B, T, seed=1)
    Tp = T - hy.start_ts
    if with_masks:
        masks_per_step = [O.make_masks(hy, B, Tp, seed=30 + st) for st in range(steps)]
    m.train()
    adam = hp.Optim["args"]["adam"]
    opt = torch.optim.Adam(m.parameters(), lr=hp.lr, betas=tuple(adam["betas"]), eps=adam["eps"])
    out = {"B": B, "T": T, "steps": steps, "lr": np.float64(hp.lr), "with_masks": int(with_masks)}
    theta0 = None
    losses, gnorms = [], []
    for st in range(steps):
        if with_masks:
            for mod_name in O.MODALITIES:
                enc = getattr(m.feature_encoder, mod_name + "_encoder", None)
                if enc is not None and masks_per_step[st][mod_name] is not None:
                    enc.dropout = _MaskFeeder(masks_per_step[st][mod_name])
        opt.zero_grad()
        loss = m(batch)[1]
        if theta0 is None:  # after the DDI of the first forward: ActNorm parameters are data dependent
            theta0 = {n: p.detach().clone() for n, p in m.named_parameters()}
        loss.backward()
        gn = torch.nn.utils.clip_grad_norm_(m.parameters(), hp.gradient_clip_val)
        opt.step()
        losses.append(float(loss))
        gnorms.append(float(gn))
        print(tag, "step", st, "loss", float(loss), "grad norm", float(gn))
    out["losses"] = np.array(losses, dtype=np.float64)
    out["grad_norms"] = np.array(gnorms, dtype=np.float64)
    names = [n for n, _ in m.named_parameters()]
    out["names"] = np.array(names)
    delta = {n: (p.detach() - theta0[n]) for n, p in m.named_parameters()}
    out["delta_l2"] = np.array([float(delta[n].double().norm()) for n in names])
    out["delta_sum"] = np.array([float(delta[n].double().sum()) for n in names])
    keep_full = names if full_tensors else [n for n in names if n.endswith(("layers.0.actnorm.logs", "layers.0.invconv.log_s", "layers.7.f.final_linear.weight",
                                                                              "layers.15.f.rnn.weight_hh", "p1_speech_encoder.encoder.weight_hh_l0",
                                                                              "layers.3.f.rnn.bias_ih"))]
    for n in keep_full:
        out["delta/" + n] = delta[n].numpy()
    for n, p in theta0.items():
        if full_tensors or ".actnorm." in n:
            out["theta0/" + n] = p.numpy()
    if full_tensors:
        for k, v in batch.items():
            out["batch/" + k] = v.numpy()
    path = os.path.join(GOLDEN, tag + ".npz")
    np.savez_compressed(path, **out)
    print(tag, "->", path, "%.1f KB" % (os.path.getsize(path) / 1024))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="")
    a = ap.parse_args()
    os.makedirs(GOLDEN, exist_ok=True)
    torch.set_num_threads(os.cpu_count())
    if a.only in ("", "small_gru"):
        run_case(small_hparams("gru"), B=6, T=12, infer_len=12, with_masks=True, full_tensors=True, tag="kat_small_gru")
    if a.only in ("", "small_lstm"):
        run_case(small_hparams("lstm"), B=6, T=12, infer_len=12, with_masks=True, full_tensors=True, tag="kat_small_lstm")
    if a.only in ("", "full"):
        run_case(load_reference_hparams(), B=64, T=80, infer_len=80, with_masks=True, full_tensors=False, tag="kat_full")
    if a.only in ("", "long"):
        run_long_sampling(load_reference_hparams(), B=16, gen_frames=750, keep=4, tag="kat_long")
    if a.only in ("", "steps"):
        run_train_steps(small_hparams("gru"), B=6, T=12, steps=3, with_masks=True, full_tensors=True, tag="kat_steps_small")
        run_train_steps(load_reference_hparams(), B=64, T=80, steps=3, with_masks=False, full_tensors=False, tag="kat_steps_full")


if __name__ == "__main__":
    main()
