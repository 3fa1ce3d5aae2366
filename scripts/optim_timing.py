"""Time of the fused clip + optimizer update over the flat parameter buffer of final_model.yaml (n = n_theta), per optimizer.

Each case is two launches (the norm pass `sumsq`, then the update) timed with CUDA events over many steps after a warm-up.  Every
case's working set (theta, gradient and its state buffers, 12 to 36 bytes per element) is larger than the 126 MB L2 of a B200, so
the update streams from HBM.  Printed per case: microseconds per update, the bytes it must move (the update's reads and writes
plus 4 bytes per element for the norm pass), the rate in GB/s, and the card's name and power limit, read in the same run.

    python scripts/optim_timing.py [--steps 200] [--warmup 20]
"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from lets_face_it_b200 import _cabi as cabi  # noqa: E402

# name, torch.optim arguments, bytes per element of the update (reads + writes)
CASES = [
    ("adam", {}, 28),                                                          # theta, m, v in and out; grad in
    ("sgd mu=0", {"momentum": 0.0}, 12),                                       # theta in and out; grad in
    ("sgd mu=0.9", {"momentum": 0.9}, 20),                                     # + buf in and out
    ("sgd nesterov", {"momentum": 0.9, "nesterov": True}, 20),
    ("rmsprop", {}, 20),                                                       # theta, square_avg in and out; grad in
    ("rmsprop centered mu=0.9", {"centered": True, "momentum": 0.9}, 36),      # + grad_avg, buf in and out
]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out or "unknown"


def launch(label, args, theta, g, bufs, hyper, n, scratch):
    L, st = cabi.lib(), cabi.stream_ptr()
    p = lambda k: bufs[k].data_ptr() if k in bufs else None
    if label == "adam":
        return L.lfi_clip_adam_dev(theta.data_ptr(), g.data_ptr(), p("m"), p("v"), n, hyper.data_ptr(), 0.9, 0.9999, 1e-8, 20.0, 1.0,
                                   scratch.data_ptr(), st)
    if label.startswith("sgd"):
        return L.lfi_clip_sgd_dev(theta.data_ptr(), g.data_ptr(), p("buf"), n, hyper.data_ptr(), args["momentum"], 0.0, 0.0,
                                  int(args.get("nesterov", False)), 20.0, 1.0, scratch.data_ptr(), st)
    return L.lfi_clip_rmsprop_dev(theta.data_ptr(), g.data_ptr(), p("sq"), p("ga"), p("buf"), n, hyper.data_ptr(), 0.99, 1e-8, 0.0,
                                  args.get("momentum", 0.0), 20.0, 1.0, scratch.data_ptr(), st)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("optim_timing.py needs a CUDA device")
    from tests.helpers import final_hparams
    from tests.kat import build_kat_model

    dev = torch.device("cuda", 0)
    n = build_kat_model(final_hparams(), dev).engine().n_theta
    gpu, power = card()
    print("%s, power limit %s; n = %d (n_theta of final_model.yaml)" % (gpu, power, n))
    gen = torch.Generator(device=dev).manual_seed(0)
    theta = torch.randn(n, device=dev, generator=gen)
    g = torch.randn(n, device=dev, generator=gen) * 1e-3
    scratch = torch.zeros(2, device=dev)
    rates = {}
    for label, args, upd_bytes in CASES:
        names = {"adam": ("m", "v")}.get(label) or (
            (("buf",) if args["momentum"] else ()) if label.startswith("sgd") else
            ("sq",) + (("ga",) if args.get("centered") else ()) + (("buf",) if args.get("momentum") else ()))
        bufs = {k: torch.zeros(n, device=dev) + (1.0 if k == "sq" else 0.0) for k in names}
        # Adam: (lr, bias corrections) of step 10; SGD: (lr, not a first step); RMSprop: (lr,)
        hyper = torch.tensor({"a": [1e-9, 0.651, 0.0316], "s": [1e-9, 0.0], "r": [1e-9]}[label[0]], device=dev)
        ws = n * (4 * (2 + len(names)))
        assert ws > 126e6, (label, ws)  # larger than L2: every pass streams from HBM
        for _ in range(a.warmup):
            cabi.check(launch(label, args, theta, g, bufs, hyper, n, scratch), label)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.steps):
            launch(label, args, theta, g, bufs, hyper, n, scratch)
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / a.steps
        moved = n * (upd_bytes + 4)
        rates[label] = moved / us / 1e3
        print("%-26s %8.1f us  %6.1f MB  %7.1f GB/s  (%.0f%% of adam's rate)" % (label, us, moved / 1e6, rates[label],
                                                                                 100 * rates[label] / rates["adam"]))
        del bufs


if __name__ == "__main__":
    main()
