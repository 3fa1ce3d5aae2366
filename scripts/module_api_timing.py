"""Time one frame, forward + backward, of two module-API calls at the final_model.yaml shapes (C 56, H 128, cond_dim 512, feature
dim 1560, B 256) on the project's kernels against the same computation in torch eager on the same GPU, with CUDA events.  One
frame = forward from a carried state, then backward of a fixed upstream gradient.
  fseq     f_seq.forward (In 28, Out 56): lfi_fseq_fwd / lfi_fseq_bwd against torch ops
  reverse  FlowStep.forward(reverse=True) (affine, LU): lfi_flowstep_rev_fwd_train / lfi_flowstep_rev_bwd, including the
           per-call W^-1 and derived-cache rebuild, against the oracle's reverse flow_step (oracle/glow_oracle.py) on the GPU

    python scripts/module_api_timing.py [--iters 200] [--warmup 20] [--rnn gru lstm] [--leg fseq reverse]

Prints one JSON line per (leg, RNN type), with the GPU name and power limit beside the times."""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from lets_face_it_b200 import _cabi  # noqa: E402
from lets_face_it_b200.glow import FlowStep, f_seq  # noqa: E402
from oracle import glow_oracle as O  # noqa: E402

In, Out, H, D, Fdim, B = 28, 56, 128, 512, 1560, 256
C = 2 * In


def eager(f, z, cond, h, c):
    """Reference f_seq.forward (models.py:204-214) in torch ops."""
    ct = F.leaky_relu(F.linear(cond, f.cond_transform[0].weight, f.cond_transform[0].bias), 0.01)
    x = torch.cat((z, ct), dim=1)
    r = f.rnn
    if f.rnn_type == "gru":
        h = torch.gru_cell(x, h, r.weight_ih, r.weight_hh, r.bias_ih, r.bias_hh)
    else:
        h, c = torch.lstm_cell(x, (h, c), r.weight_ih, r.weight_hh, r.bias_ih, r.bias_hh)
    fl = f.final_linear
    return F.linear(h, fl.weight, fl.bias) * torch.exp(fl.logs * fl.logscale_factor)


def time_ms(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(iters):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / iters


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                           timeout=30)
        power = q.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def reverse_leg(rnn, a, dev, g, name, power):
    torch.manual_seed(0)
    step = FlowStep(C, H, D, flow_permutation="invconv", flow_coupling="affine", LU_decomposed=True, scale_eps=1e-4,
                    feature_encoder_dim=Fdim, glow_rnn_type=rnn).to(dev)
    with torch.no_grad():
        for n, p in step.named_parameters():
            if "final_linear" in n or "actnorm" in n:
                p.normal_(0, 0.15, generator=g)
    step.actnorm.inited = True
    hy = O.Hyper(C=C, K=1, H=H, D=D, rnn_type=rnn, scale_eps=1e-4, actnorm_scale=1.0, LU=True, coupling="affine",
                 hist={m: 1 for m in O.MODALITIES}, enc={m: "none" for m in O.MODALITIES}, enc_hidden={m: 0 for m in O.MODALITIES},
                 in_dim={m: 1 for m in O.MODALITIES}, dropout={m: 0.0 for m in O.MODALITIES})
    P = {"glow.flow.layers.0." + k: v.detach().clone().requires_grad_(v.is_floating_point() and not k.endswith((".p", ".sign_s")))
         for k, v in step.state_dict().items()}
    z = torch.randn(B, C, device=dev, generator=g).requires_grad_(True)
    cond = torch.randn(B, Fdim, device=dev, generator=g).requires_grad_(True)
    h0 = torch.randn(B, H, device=dev, generator=g)
    c0 = torch.randn(B, H, device=dev, generator=g) if rnn == "lstm" else None
    R, Rl = torch.randn(B, C, device=dev, generator=g), torch.randn(B, device=dev, generator=g)
    ld0 = torch.zeros(B, device=dev)

    def ours():
        step.f.hidden, step.f.cell = h0, c0
        y, ld = step(z, cond, ld0, reverse=True)
        ((y * R).sum() + (ld * Rl).sum()).backward()

    def oracle_fwd():
        with torch.device(dev):  # the oracle builds its LU masks with default-device factories
            return O.flow_step(P, hy, 0, z, cond, ld0, True, {0: h0 if c0 is None else (h0, c0)})

    def ref():
        y, ld = oracle_fwd()
        ((y * R).sum() + (ld * Rl).sum()).backward()

    with torch.no_grad():
        step.f.hidden, step.f.cell = h0, c0
        diff = float((step(z, cond, ld0, reverse=True)[0] - oracle_fwd()[0]).abs().max())
    L = _cabi.lib()
    n0 = L.lfi_launch_count()
    ours()
    torch.cuda.synchronize()
    launches = L.lfi_launch_count() - n0
    t_ours = time_ms(ours, a.iters, a.warmup)
    t_ref = time_ms(ref, a.iters, a.warmup)
    t_ours2 = time_ms(ours, a.iters, a.warmup)
    print(json.dumps({"leg": "flowstep_reverse", "rnn": rnn, "B": B, "C": C, "H": H, "D": D, "F": Fdim,
                      "fwd_bwd_ms_per_frame": [round(t_ours, 4), round(t_ours2, 4)], "torch_eager_oracle_ms_per_frame": round(t_ref, 4),
                      "library_launches_per_frame": launches, "max_abs_diff_vs_oracle": diff, "gpu": name, "power_limit": power}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rnn", nargs="+", default=["gru", "lstm"])
    ap.add_argument("--leg", nargs="+", default=["fseq", "reverse"], choices=["fseq", "reverse"])
    a = ap.parse_args()
    dev = "cuda:0"
    name, power = gpu_info()
    g = torch.Generator(device=dev).manual_seed(0)
    if "reverse" in a.leg:
        for rnn in a.rnn:
            reverse_leg(rnn, a, dev, g, name, power)
    if "fseq" not in a.leg:
        return
    for rnn in a.rnn:
        torch.manual_seed(0)
        f = f_seq(In, Out, H, D, Fdim, rnn).to(dev)
        with torch.no_grad():
            for p in (f.final_linear.weight, f.final_linear.bias, f.final_linear.logs):
                p.normal_(0, 0.1, generator=g)
        z = torch.randn(B, In, device=dev, generator=g).requires_grad_(True)
        cond = torch.randn(B, Fdim, device=dev, generator=g).requires_grad_(True)
        h0 = torch.randn(B, H, device=dev, generator=g)
        c0 = torch.randn(B, H, device=dev, generator=g) if rnn == "lstm" else None
        R = torch.randn(B, Out, device=dev, generator=g)

        def ours():
            f.hidden, f.cell = h0, c0
            f(z, cond).backward(R)

        def ref():
            eager(f, z, cond, h0, c0 if c0 is not None else torch.zeros_like(h0)).backward(R)

        f.hidden, f.cell = h0, c0
        with torch.no_grad():
            diff = float((f(z, cond) - eager(f, z, cond, h0, c0 if c0 is not None else torch.zeros_like(h0))).abs().max())
        L = _cabi.lib()
        n0 = L.lfi_launch_count()
        ours()
        torch.cuda.synchronize()
        launches = L.lfi_launch_count() - n0
        t_ours = time_ms(ours, a.iters, a.warmup)
        t_ref = time_ms(ref, a.iters, a.warmup)
        t_ours2 = time_ms(ours, a.iters, a.warmup)  # second pass: the spread of the measurement
        print(json.dumps({"rnn": rnn, "B": B, "In": In, "Out": Out, "H": H, "D": D, "F": Fdim, "fwd_bwd_ms_per_frame": [round(t_ours, 4), round(t_ours2, 4)],
                          "torch_eager_ms_per_frame": round(t_ref, 4), "library_launches_per_frame": launches, "max_abs_diff_vs_eager": diff,
                          "gpu": name, "power_limit": power}))


if __name__ == "__main__":
    main()
