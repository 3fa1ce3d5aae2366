"""Time and memory of SeqGlow.evaluate (time-chunked, no-grad likelihood) at final_model.yaml shapes, B = 256, bf16x3.

1. T = 80: the no-grad `forward` (training workspace) against `evaluate`, alternating, --calls calls each after a warm-up, timed
   with CUDA events; and the peak allocation of one call of each (max_memory_allocated after reset_peak_memory_stats, with
   the other path's workspace released: model, batch, the call's workspace and outputs).
2. `evaluate` at T = 24 + {560, 2000, 7500}: ms per scored frame (mean of --long-calls calls after one warm-up call), peak
   allocation of one call, and what lfi_train_ws_bytes says the no-grad `forward` of the same shape would need (computed only).

Prints one JSON line per measurement, with the card's name and power limit read in the same run.

    python scripts/eval_timing.py [--calls 20] [--long-calls 3] [--out DIR]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from lets_face_it_b200 import _cabi as cabi  # noqa: E402
from tests.helpers import final_hparams  # noqa: E402
from tests.kat import build_kat_model, kat_batch, to_device  # noqa: E402

B = 256


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out or "unknown"


def timed(fn, n):
    """Mean ms of fn() over n calls, CUDA events around each call."""
    ms = 0.0
    for _ in range(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms += e0.elapsed_time(e1)
    return ms / n


def peak(model, fn):
    """max_memory_allocated over one call of fn, with the engine's workspaces released first: the model, the batch, the
    call's own workspace and its outputs."""
    model._engine._ws.clear()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--long-calls", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON lines to DIR/eval_timing.jsonl")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "eval_timing.py measures on a CUDA device"
    name, power = card()
    hp = final_hparams()
    m = build_kat_model(hp, "cuda:0")
    m.glow.set_actnorm_init(True)
    m.gemm_mode = cabi.GEMM_BF16X3
    m.eval()
    eng = m.engine()
    L = cabi.lib()
    rows = []

    def emit(rec):
        rec.update(card=name, power_limit=power, B=B, mode="bf16x3")
        print(json.dumps(rec), flush=True)
        rows.append(rec)

    batch = to_device(kat_batch(hp, B, 80, seed=5), "cuda:0")

    def fwd():
        with torch.no_grad():
            m(batch)

    def ev():
        m.evaluate(batch)

    for _ in range(3):
        fwd()
        ev()
    t_f = t_e = 0.0
    for _ in range(args.calls):  # alternating, one call of each per round
        t_f += timed(fwd, 1)
        t_e += timed(ev, 1)
    p_f, p_e = peak(m, fwd), peak(m, ev)
    emit(dict(case="T=80", T=80, calls=args.calls, forward_ms=t_f / args.calls, evaluate_ms=t_e / args.calls,
              forward_peak_bytes=p_f, evaluate_peak_bytes=p_e, chunk=eng.eval_chunk(B, 80),
              train_ws_bytes=L.lfi_train_ws_bytes(ctypes.byref(eng.shape), B, 80, cabi.GEMM_BF16X3),
              eval_ws_bytes=L.lfi_eval_ws_bytes(ctypes.byref(eng.shape), B, 80, eng.eval_chunk(B, 80), cabi.GEMM_BF16X3),
              evaluate_ms_per_frame=t_e / args.calls / 56))

    for Tp in (560, 2000, 7500):
        T = 24 + Tp
        lb = to_device(kat_batch(hp, B, T, seed=6), "cuda:0")
        run = lambda: m.evaluate(lb)
        run()
        ms = timed(run, args.long_calls)
        pk = peak(m, run)
        chunk = eng.eval_chunk(B, T)
        emit(dict(case="long", T=T, calls=args.long_calls, evaluate_ms=ms, evaluate_ms_per_frame=ms / Tp, evaluate_peak_bytes=pk,
                  chunk=chunk, eval_ws_bytes=L.lfi_eval_ws_bytes(ctypes.byref(eng.shape), B, T, chunk, cabi.GEMM_BF16X3),
                  train_ws_bytes_not_run=L.lfi_train_ws_bytes(ctypes.byref(eng.shape), B, T, cabi.GEMM_BF16X3)))
        del lb
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "eval_timing.jsonl"), "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
