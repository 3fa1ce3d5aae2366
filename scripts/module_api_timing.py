"""Time f_seq.forward + backward per frame at the final_model.yaml shapes (In 28, Out 56, H 128, cond_dim 512, feature dim
1560, B 256) on the project's kernels (lfi_fseq_fwd / lfi_fseq_bwd) against the same computation in torch eager on the same
GPU, with CUDA events.  One frame = forward from a carried state, then backward of a fixed upstream gradient.

    python scripts/module_api_timing.py [--iters 200] [--warmup 20] [--rnn gru lstm]

Prints one JSON line per RNN type, with the GPU name and power limit beside the times."""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from lets_face_it_b200 import _cabi  # noqa: E402
from lets_face_it_b200.glow import f_seq  # noqa: E402

In, Out, H, D, Fdim, B = 28, 56, 128, 512, 1560, 256


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rnn", nargs="+", default=["gru", "lstm"])
    a = ap.parse_args()
    dev = "cuda:0"
    name, power = gpu_info()
    g = torch.Generator(device=dev).manual_seed(0)
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
