"""Time the training backward with and without input gradients at the final_model.yaml shapes (B 256, T 80, bf16x3, frame dropout
on): lfi_seq_train_bwd against lfi_seq_train_bwd_dx (every stream's gradient wanted) on the same forward stash, and SeqGlow.forward
+ loss.backward() with and without batch tensors that require grad.  CUDA events; the two variants alternate in blocks so that a
drift of the card's clocks hits both.

    python scripts/seq_dx_timing.py [--iters 20] [--rounds 5] [--warmup 3]

Prints one JSON line with the GPU name and power limit beside the times (medians over the rounds, ms per call)."""
import argparse
import ctypes
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from lets_face_it_b200 import _cabi  # noqa: E402
from lets_face_it_b200.hparams import load_hparams  # noqa: E402
from oracle import glow_oracle as O  # noqa: E402
from scripts.encoder_api_timing import gpu_info, time_ms  # noqa: E402
from tests.kat import build_kat_model  # noqa: E402

B, T = 256, 80


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("seq_dx_timing.py needs a CUDA device")
    dev = "cuda:0"
    hp = load_hparams()
    hy = O.Hyper.from_hparams(hp)
    m = build_kat_model(hp, dev).train()
    m.glow.set_actnorm_init(True)
    m.gemm_mode = _cabi.GEMM_BF16X3
    Tp = T - hy.start_ts
    batch = {k: v.to(dev) for k, v in O.synthetic_batch(hy, B, T, seed=1).items()}
    masks = {k: (v.to(dev) if v is not None else None) for k, v in O.make_masks(hy, B, Tp, seed=3).items()}
    m.injected_masks = masks
    eng = m.engine()

    z, nll = eng.train_forward(batch, masks)
    dnll = torch.full_like(nll, 1.0 / nll.numel())
    g = eng.new_flat_grad()
    dx = [torch.empty(B, T, eng.shape.dim[i], device=dev) if eng.shape.hist[i] > 0 else None for i in range(_cabi.NMOD)]

    def bwd_plain():
        eng.train_backward(z, dnll, g)

    def bwd_dx():
        eng.train_backward(z, dnll, g, dx=dx)

    def step(b):
        _, loss, _ = m(b)
        loss.backward()

    def step_plain():
        step(batch)

    xs = {k: v.clone().requires_grad_(True) for k, v in batch.items()}

    def step_dx():
        for v in xs.values():
            v.grad = None
        step(xs)

    runs = {"bwd_plain": bwd_plain, "bwd_dx": bwd_dx, "step_plain": step_plain, "step_dx": step_dx}
    times = {k: [] for k in runs}
    for fn in runs.values():
        time_ms(fn, 1, a.warmup)
    for _ in range(a.rounds):
        for k, fn in runs.items():
            times[k].append(time_ms(fn, a.iters, 0))
    out = {"%s_ms" % k: round(statistics.median(v), 4) for k, v in times.items()}
    out.update({"%s_spread_ms" % k: [round(min(v), 4), round(max(v), 4)] for k, v in times.items()})
    out["dx_ws_bytes"] = int(_cabi.lib().lfi_train_dx_ws_bytes(ctypes.byref(eng.shape), B, T, _cabi.GEMM_BF16X3))
    name, power = gpu_info()
    out.update(gpu=name, power_limit=power, B=B, T=T, mode="bf16x3", iters=a.iters, rounds=a.rounds)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
