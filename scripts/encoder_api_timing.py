"""Time one SeqGlow.create_conditioning forward + backward at the final_model.yaml shapes (B 256; p1_face window 5 x 56, GRU
encoders p2_face 24 x 56 -> 256, p1_speech 2 x 30 -> 128, p2_speech 16 x 30 -> 256) on the project's kernels
(lfi_feature_encode_fwd_train / lfi_feature_encode_bwd) in each gemm mode, against the reference's FeatureEncoder in torch eager
(nn.GRU per modality, autograd) on the same GPU, with CUDA events.  The upstream gradient is fixed; the windows require grad.

    python scripts/encoder_api_timing.py [--iters 50] [--warmup 5]

Prints one JSON line with the GPU name and power limit beside the times."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from lets_face_it_b200 import _cabi  # noqa: E402
from lets_face_it_b200.hparams import load_hparams  # noqa: E402
from oracle import glow_oracle as O  # noqa: E402
from tests.kat import build_kat_model  # noqa: E402

B = 256


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
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("encoder_api_timing.py needs a CUDA device")
    dev = "cuda:0"
    hp = load_hparams()
    hy = O.Hyper.from_hparams(hp)
    m = build_kat_model(hp, dev)
    T = hy.start_ts + 1
    data = {k: v.to(dev).requires_grad_(True) for k, v in O.synthetic_batch(hy, B, T, seed=1).items()}
    R = torch.randn(B, hy.F, device=dev)
    t = hy.start_ts
    out = {}

    def ours():
        cond = m.create_conditioning(data, t, None, data["p1_face"])
        (cond * R).sum().backward()

    for name, mode in (("fp32", _cabi.GEMM_FP32), ("bf16x3", _cabi.GEMM_BF16X3), ("bf16", _cabi.GEMM_BF16)):
        m.gemm_mode = mode
        out["ours_%s_ms" % name] = time_ms(ours, a.iters, a.warmup)

    # reference FeatureEncoder.forward (models.py:55-80, 127-145) in torch eager: one cuDNN nn.GRU per GRU modality
    grus = {}
    for mod in O.MODALITIES:
        g = m.feature_encoder.gru_of(mod)
        if g is not None:
            ref = torch.nn.GRU(g.input_size, g.hidden_size, batch_first=True).to(dev)
            with torch.no_grad():
                for n in ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0"):
                    getattr(ref, n).copy_(getattr(g, n))
            grus[mod] = ref

    def eager():
        parts = []
        for mod in O.MODALITIES:
            h = hy.hist[mod]
            if not h:
                continue
            win = data[mod][:, t - h:t] if mod == "p1_face" else data[mod][:, t - h + 1:t + 1]
            if mod in grus:
                seq, hn = grus[mod](win)
                parts.append(torch.cat([seq[:, -1], hn[0]], dim=1))
            else:
                parts.append(win.reshape(B, -1))
        (torch.cat(parts, dim=1) * R).sum().backward()

    out["torch_eager_gru_ms"] = time_ms(eager, a.iters, a.warmup)
    name, power = gpu_info()
    out.update(gpu=name, power_limit=power, B=B, iters=a.iters)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
