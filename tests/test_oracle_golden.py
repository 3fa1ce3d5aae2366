"""CPU: pins oracle/glow_oracle.py to vectors produced by the unmodified reference
(oracle/make_golden.py), and — where LFI_REFERENCE_ROOT names a checkout of it — to the live reference."""
import numpy as np
import pytest
import torch

from oracle import glow_oracle as O
from tests.helpers import golden_batch, golden_params, load_golden, relerr, small_hparams


@pytest.mark.parametrize("rnn", ["gru", "lstm"])
def test_oracle_forward_matches_reference_vectors(rnn):
    g = load_golden("kat_small_" + rnn)
    hy = O.Hyper.from_hparams(small_hparams(rnn))
    P, batch = golden_params(g), golden_batch(g)
    with torch.no_grad():
        z, nll, loss = O.seq_forward(P, hy, batch)
    assert relerr(z, g["z"]) < 2e-6
    assert relerr(nll, g["nll"]) < 1e-6
    assert abs(float(loss) - float(g["loss"][0])) < 1e-4 * abs(float(g["loss"][0]))


@pytest.mark.parametrize("rnn", ["gru", "lstm"])
def test_oracle_sampling_and_invert_match_reference_vectors(rnn):
    g = load_golden("kat_small_" + rnn)
    hy = O.Hyper.from_hparams(small_hparams(rnn))
    P, batch = golden_params(g), golden_batch(g)
    data = dict(batch)
    data["p1_face"] = torch.zeros(int(g["B"]), hy.start_ts, hy.C)
    L = int(g["infer_len"])
    x0 = O.seq_inference(P, hy, data, L, eps=0.0, noise=torch.zeros(L - hy.start_ts, int(g["B"]), hy.C))
    assert relerr(x0, g["x_eps0"]) < 5e-6
    x1 = O.seq_inference(P, hy, data, L, noise=torch.from_numpy(g["noise"]))
    assert relerr(x1, g["x_noise"]) < 5e-6
    rec, _ = O.seq_invert(P, hy, list(torch.from_numpy(g["z"])), batch)
    assert relerr(rec, g["rec"]) < 5e-5


@pytest.mark.parametrize("rnn", ["gru", "lstm"])
def test_oracle_backward_matches_reference_vectors(rnn):
    g = load_golden("kat_small_" + rnn)
    hy = O.Hyper.from_hparams(small_hparams(rnn))
    P = O.clone_params(golden_params(g), requires_grad=True)
    batch = golden_batch(g)
    _, _, loss = O.seq_forward(P, hy, batch)
    loss.backward()
    for n in g["grad_names"]:
        ref = torch.from_numpy(g["grad/" + str(n)])
        got = P["" + str(n)].grad.reshape(ref.shape)
        assert relerr(got, ref) < 2e-4, n


@pytest.mark.parametrize("rnn", ["gru", "lstm"])
def test_oracle_dropout_masks_match_reference_vectors(rnn):
    g = load_golden("kat_small_" + rnn)
    hy = O.Hyper.from_hparams(small_hparams(rnn))
    P = O.clone_params(golden_params(g), requires_grad=True)
    batch = golden_batch(g)
    masks = O.make_masks(hy, int(g["B"]), int(g["T"]) - hy.start_ts, seed=3)
    z, nll, loss = O.seq_forward(P, hy, batch, masks)
    loss.backward()
    assert relerr(z.detach(), g["masked_z"]) < 2e-6
    assert relerr(nll.detach(), g["masked_nll"]) < 1e-6
    for n in g["grad_names"]:
        ref = torch.from_numpy(g["masked_grad/" + str(n)])
        assert relerr(P[str(n)].grad.reshape(ref.shape), ref) < 2e-4, n


def test_oracle_ddi_matches_reference_vectors():
    """ActNorm data-dependent init (modules.py:32-43): start from the pre-DDI parameters."""
    g = load_golden("kat_small_gru")
    hy = O.Hyper.from_hparams(small_hparams("gru"))
    P, batch = golden_params(g), golden_batch(g)
    for k in list(P):
        if ".actnorm." in k:
            P[k] = torch.zeros_like(P[k])
    O.ddi_init(P, hy, batch)
    for k in P:
        if ".actnorm." in k:
            assert relerr(P[k], g["param/" + k]) < 1e-5, k


# ------------------------------------------------------------------------------------------------ round 2: the benchmarked paths
def _full_kat_params(g):
    """KAT parameters of final_model.yaml (constructor + seeds, tests/kat.py) with the reference's post-DDI ActNorm values."""
    from tests.helpers import final_hparams
    from tests.kat import build_kat_model, oracle_params_from

    hp = final_hparams()
    P = oracle_params_from(build_kat_model(hp))
    for k in g.files:
        if k.startswith("param/") and ".actnorm." in k:
            P[k[len("param/"):]] = torch.from_numpy(g[k])
    return hp, P


def test_oracle_masked_full_kat_matches_reference_vectors():
    """final_model.yaml with the frame-dropout masks injected (models.py:56-58), first 8 of the 64 KAT sequences:
    z and NLL of the live reference (kat_full.npz: masked_*)."""
    from tests.kat import kat_batch

    g = load_golden("kat_full")
    hp, P = _full_kat_params(g)
    hy = O.Hyper.from_hparams(hp)
    B, T, S = int(g["B"]), int(g["T"]), 8
    batch = {k: v[:S] for k, v in kat_batch(hp, B, T).items()}
    masks = O.make_masks(hy, B, T - hy.start_ts, seed=3)
    masks = {k: (v[:, :S].contiguous() if v is not None else None) for k, v in masks.items()}
    with torch.no_grad():
        z, nll, _ = O.seq_forward(P, hy, batch, masks)
    assert relerr(z, g["masked_z_head"]) < 5e-6
    assert relerr(nll, g["masked_nll"][:, :S]) < 1e-6


def test_oracle_long_horizon_sampling_matches_reference_vectors():
    """750 generated frames at temperature 0.7 (BASELINE.json configs[3] horizon), 2 of the stored sequences: the oracle's
    frame loop tracks the live reference over the whole horizon (no drift)."""
    g = load_golden("kat_long")
    hp, P = _full_kat_params(g)
    hy = O.Hyper.from_hparams(hp)
    B, Tg, S = int(g["B"]), int(g["gen_frames"]), 2
    seq_len = hy.start_ts + Tg
    data = {k: v[:S] for k, v in O.synthetic_batch(hy, B, seq_len, seed=5).items()}
    data["p1_face"] = torch.zeros(S, hy.start_ts, hy.C)
    noise = torch.randn(Tg, B, hy.C, generator=torch.Generator().manual_seed(21)) * 0.7
    with torch.no_grad():
        x = O.seq_inference(P, hy, data, seq_len, noise=noise[:, :S].contiguous())
    ref = torch.from_numpy(g["x_head"][:S])
    per_frame = (x - ref).abs().amax(dim=(0, 2)) / ref.abs().max()
    assert float(per_frame.max()) < 2e-5, (int(per_frame.argmax()), float(per_frame.max()))
    assert float(per_frame[-250:].max()) < 3 * float(per_frame[:250].max()) + 1e-6


def test_oracle_three_optimizer_steps_match_reference_vectors():
    """Three steps of (forward with that step's masks, backward, clip_grad_norm_ 20, torch.optim.Adam) on the oracle's
    parameters against the same three steps of the live reference (kat_steps_small.npz)."""
    g = load_golden("kat_steps_small")
    hp = small_hparams("gru")
    hy = O.Hyper.from_hparams(hp)
    from tests.kat import build_kat_model, oracle_params_from

    P = O.clone_params(oracle_params_from(build_kat_model(hp)), requires_grad=True)
    batch = golden_batch(g)
    B, T, steps = int(g["B"]), int(g["T"]), int(g["steps"])
    adam = hp.Optim["args"]["adam"]
    theta0 = None
    for st in range(steps):
        masks = O.make_masks(hy, B, T - hy.start_ts, seed=30 + st)
        if st == 0:
            O.ddi_init(P, hy, batch, masks)  # replaces the ActNorm leaves: collect the leaves afterwards
            theta0 = {k: v.detach().clone() for k, v in P.items()}
            leaves = [v for v in P.values() if v.requires_grad]
            opt = torch.optim.Adam(leaves, lr=hp.lr, betas=tuple(adam["betas"]), eps=adam["eps"])
        opt.zero_grad()
        _, _, loss = O.seq_forward(P, hy, batch, masks)
        loss.backward()
        gn = torch.nn.utils.clip_grad_norm_(leaves, hp.gradient_clip_val)
        opt.step()
        assert abs(float(loss) - float(g["losses"][st])) < 1e-5 * abs(float(g["losses"][st])), st
        assert abs(float(gn) - float(g["grad_norms"][st])) < 1e-4 * float(g["grad_norms"][st]), st
    for n in g["names"]:
        n = str(n)
        ref = torch.from_numpy(g["delta/" + n]).double()
        got = (P[n].detach() - theta0[n]).double().reshape(ref.shape)
        assert float((got - ref).norm()) <= 0.02 * float(ref.norm()) + 1e-12, n


def test_packaged_final_model_yaml_matches_values_the_reference_recorded():
    """The packaged final_model.yaml against what the reference's runs on its own final_model.yaml stored in the golden
    vectors: the learning rate of its optimizer steps (kat_steps_full), the face-parameter split of its output side and the
    modalities its mismatched-NLL probe shuffles (kat_post).  The shape-bearing Conditioning / Glow values are pinned by
    the bit-identical parameters test_cabi_symbols.py::test_dropin_constructor_reproduces_reference_parameters builds."""
    from lets_face_it_b200.glow.utils import get_mismatched_modalities
    from lets_face_it_b200.hparams import load_hparams

    hp = load_hparams()
    steps, post = load_golden("kat_steps_full"), load_golden("kat_post")
    assert hp.lr == float(steps["lr"])
    assert [hp.Data[k] for k in ("expression_dim", "jaw_dim", "neck_dim")] == [int(v) for v in post["data_dims"]]
    mods, name = get_mismatched_modalities(hp)
    assert mods == [str(m) for m in post["mismatched_modalities"]] and name == str(post["mismatched_name"])


@pytest.mark.reference
def test_reference_yaml_files_load_unchanged():
    """The reference's own hparams files (code/glow_pytorch/hparams/*.yaml, 159 lines each) load through
    `lets_face_it_b200.hparams.load_hparams` and build the drop-in SeqGlow; for final_model.yaml the result has exactly the
    shapes of the packaged subset (runs only where LFI_REFERENCE_ROOT names a checkout of the reference)."""
    import os

    from lets_face_it_b200.glow import SeqGlow
    from lets_face_it_b200.hparams import load_hparams
    from oracle.ref_shim import REF_YAML_DIR

    ours = load_hparams()
    for name in ("final_model.yaml", "no_face.yaml", "no_speech.yaml", "no_nll_trick.yaml"):
        path = os.path.join(REF_YAML_DIR, name)
        if not os.path.isfile(path):
            continue
        hp = load_hparams(path)
        torch.manual_seed(0)
        np.random.seed(0)
        m = SeqGlow(hp)
        assert m.feature_encoder.dim == hp.Conditioning["p1_face"]["dim"] * hp.Conditioning["p1_face"]["history"] + sum(
            2 * hp.Conditioning[k]["hidden_dim"] for k in ("p2_face", "p1_speech", "p2_speech") if hp.Conditioning[k]["history"])
        if name == "final_model.yaml":
            for sec in ("Conditioning", "Glow", "Data"):
                for k, v in getattr(ours, sec).items():
                    ref = getattr(hp, sec)[k]
                    if isinstance(v, dict):
                        for kk, vv in v.items():
                            assert ref[kk] == vv, (sec, k, kk)
                    else:
                        assert ref == v, (sec, k)
            assert hp.lr == ours.lr and hp.gradient_clip_val == ours.gradient_clip_val and hp.batch_size == ours.batch_size
            assert hp.Optim["args"]["adam"] == ours.Optim["args"]["adam"]
            assert hp.Optim["Schedule"]["args"]["step"] == ours.Optim["Schedule"]["args"]["step"]
