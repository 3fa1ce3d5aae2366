#!/usr/bin/env python
"""Benchmark of the conditional-Glow hot path (BASELINE.json metric: train frames/sec, final_model.yaml).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--gemm fp32|bf16x3|bf16] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = one optimizer step (forward + NLL + backward + clip_grad_norm 20 + Adam) on a batch of 256 synthetic
sequences per GPU, T=80 (56 trained frames per sequence) — BASELINE.json configs[1]; for N>1 every rank takes its own
256 sequences (weak scaling) and the flat fp32 gradient is all-reduced over NCCL.  Prints ONE JSON line (rank 0).

`--impl reference` times the reference algorithm's CPU path (the oracle port: the reference is pure Python/PyTorch,
there is nothing to compile) on the host cores, on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_FRAME_TRAIN = 127.15e6   # canonical (folded) training FLOP per frame per sequence, SURVEY.md §8(d)
FLOP_PER_FRAME_FWD = 42.38e6
T_TRAIN, START_TS = 80, 24


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--gemm", default=os.environ.get("LFI_GEMM", "bf16x3"), choices=["fp32", "bf16x3", "bf16"],
                    help="contraction mode: bf16x3 = error-compensated split-bf16 on tcgen05 (fp32-grade, the parity mode), "
                         "bf16 = plain bf16 operands (looser stated bound), fp32 = FFMA tiles")
    ap.add_argument("--sample-seqs", type=int, default=1024, help="concurrent sequences per GPU of the sampling leg")
    ap.add_argument("--sample-frames", type=int, default=750, help="generated frames per sequence (30 s at 25 fps)")
    ap.add_argument("--batch", type=int, default=256, help="sequences per GPU")
    ap.add_argument("--strong", action="store_true",
                    help="strong scaling (secondary number, SURVEY.md section 8(d) config 3): the GLOBAL batch stays --batch, each GPU takes batch / N")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-batch", type=int, default=256, help="sequences per step of the CPU reference arm (default: the same B=256 step as our arm)")
    ap.add_argument("--no-sample", action="store_true")
    ap.add_argument("--no-bf16", action="store_true", help="skip the secondary bf16-mode timing")
    ap.add_argument("--variant", default="final", choices=["final", "wide-lstm", "wide-gru"],
                    help="final = final_model.yaml (the headline); wide-* = BASELINE.json configs[4]: 2x flow depth (K=32), "
                         "2x hidden size (H=256), LSTM or GRU coupling cell")
    ap.add_argument("--ncu-step", action="store_true",
                    help="profiling helper: warm up, then run ONE step between cudaProfilerStart/Stop and exit "
                         "(use with ncu --profile-from-start off); prints no bench line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed training step returned as DIR/<name>.npy: loss, "
                         "grad_norm and params (a fixed sample of the updated parameters); inputs and seeds do not change "
                         "between runs, so two builds can be compared output for output (bench_outputs/<build> in the "
                         "checkout is ignored by git)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "ours" or a.ncu_step):
        ap.error("--dump-outputs writes the outputs of the timed GPU training step: not with --impl reference or --ncu-step")
    return a


DUMP_PARAMS = 1 << 22   # parameters written by --dump-outputs (16 MB as float32; the final model has 17.6 M)


def dump_outputs(out_dir, model, trainer, loss):
    """What a caller of Trainer.step holds after the last timed step: its loss, the gradient norm the step clipped with, and
    the updated parameters (the step writes them in place), flattened in `named_parameters` order.  Larger models are
    sampled at DUMP_PARAMS positions drawn from a fixed seed, in ascending order."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    params = torch.cat([p.detach().reshape(-1) for _, p in model.named_parameters()])
    if params.numel() > DUMP_PARAMS:
        pick = torch.randperm(params.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_PARAMS].sort().values
        params = params[pick.to(params.device)]
    out = {"loss": np.float64(loss.item()), "grad_norm": np.float64(trainer.grad_norm().item()),
           "params": params.float().cpu().numpy()}
    for name, v in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), v)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("bf16_tflops_sustained", 1369.2), d.get("bf16_tflops", 1630.4), d.get("hbm_gbs", 6548.8), "measured"
    return 1400.0, 1590.0, 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def wait_first(self, timeout=4.0):
        """Blocks until nvidia-smi has written its first poll (it needs a few hundred ms to start: a short warm-up + timed
        region would otherwise be over before the first sample)."""
        if self.proc is None:
            return
        t0 = time.time()
        while time.time() - t0 < timeout:
            try:
                if os.path.getsize(self.path) > 0:
                    return
            except OSError:
                return
            time.sleep(0.02)

    def stop(self, window=None):
        """window = (t0, t1) host epoch seconds of the timed region: only samples inside it are used (the sampler is started
        before the warm-up so that nvidia-smi is already running when the region begins)."""
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        rows = []  # (timestamp or None, sm, max, reasons)
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    smv, mxv = float(f[1]), float(f[2])
                except ValueError:
                    continue
                rs = {name for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9])
                      if v.lower().startswith("active")}
                rows.append((ts, smv, mxv, rs))
            os.unlink(self.path)
        except Exception:
            pass
        sel, note = rows, None
        if window is not None and rows:
            # samples inside the timed region; a short region (10 steps ~ 0.12 s) can fall between two 50 ms polls when several
            # ranks query at once, so the margin widens (the GPU is under the same load right before / after: warm-up, e2e leg)
            for margin in (0.05, 0.3, 1.0):
                sel = [r for r in rows if window[0] - margin <= r[0] <= window[1] + margin]
                if sel:
                    note = None if margin == 0.05 else "no poll inside the timed region: samples within %.1f s of it" % margin
                    break
            if not sel:
                mid = 0.5 * (window[0] + window[1])
                sel, note = [min(rows, key=lambda r: abs(r[0] - mid))], "nearest poll to the timed region"
        if sel:
            sm = sorted(r[1] for r in sel)
            reasons = set().union(*[r[3] for r in sel])
            out = {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(r[2] for r in sel), "reasons": sorted(reasons), "samples": len(sel)}
            if note:
                out["note"] = note
        return out


def make_batch(hy, B, T, seed, pin=False):
    import torch
    from oracle import glow_oracle as O  # only for the seeded synthetic-input recipe (SURVEY.md §8(d))

    b = O.synthetic_batch(hy, B, T, seed)
    if pin:
        b = {k: v.pin_memory() for k, v in b.items()}
    return b


# ----------------------------------------------------------------------------------------------------------------
def cpu_reference_step_fn(hp, B, T):
    """The reference algorithm on the host cores (oracle port): forward + NLL + backward + clip 20 + Adam."""
    import torch
    from oracle import glow_oracle as O
    from tests.kat import build_kat_model, oracle_params_from

    torch.set_num_threads(os.cpu_count() or 1)
    hy = O.Hyper.from_hparams(hp)
    m = build_kat_model(hp)
    P = O.clone_params(oracle_params_from(m), requires_grad=True)
    del m
    batch = O.synthetic_batch(hy, B, T, seed=1)
    O.ddi_init(P, hy, batch)
    leaves = [v for v in P.values() if v.requires_grad]
    opt = torch.optim.Adam(leaves, lr=hp.lr, betas=tuple(hp.Optim["args"]["adam"]["betas"]), eps=hp.Optim["args"]["adam"]["eps"])
    masks = O.make_masks(hy, B, T - hy.start_ts, seed=3)

    def step():
        opt.zero_grad(set_to_none=True)
        _, _, loss = O.seq_forward(P, hy, batch, masks)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(leaves, hp.gradient_clip_val)
        opt.step()
        return float(loss)

    return step, B * (T - hy.start_ts)


def run_reference(a):
    import torch
    from lets_face_it_b200.hparams import load_hparams

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    hp = load_hparams()
    Bs = a.ref_batch
    step, frames = cpu_reference_step_fn(hp, Bs, T_TRAIN)
    for _ in range(a.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        step()
    dt = time.perf_counter() - t0
    v = frames * a.steps / dt
    cores = torch.get_num_threads()
    sample = "oracle port (torch CPU fp32), %d sequences x %d frames per step, fwd+bwd+clip+Adam, dropout masks on" % (Bs, T_TRAIN - START_TS)
    print(json.dumps({
        "impl": "reference", "metric": "train frames/sec", "value": v, "unit": "frames/s", "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * dt / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        # the same workload string and batch as our arm (run_ours): the same B = 256 step, timed on the host cores
        "config": {"workload": "final_model.yaml training step (fwd+NLL+bwd+clip20+Adam), B=%d sequences/GPU, T=80 (56 trained "
                               "frames/seq), frame dropout on" % Bs,
                   "global_batch": Bs, "gemm_mode": "fp32 (torch CPU)", "parallelism": "cpu%d" % cores},
        "cpu_baseline": {"value": v, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ----------------------------------------------------------------------------------------------------------------
def run_ours(a):
    import torch
    import torch.distributed as dist

    from lets_face_it_b200 import _cabi as cabi
    from lets_face_it_b200.hparams import load_hparams
    from lets_face_it_b200.train import HostFeed, Trainer
    from oracle import glow_oracle as O
    from tests.kat import build_kat_model

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    hp = load_hparams()
    if a.variant != "final":
        hp.Glow["K"] = 32
        hp.Glow["hidden_channels"] = 256
        hp.Glow["rnn_type"] = "lstm" if a.variant == "wide-lstm" else "gru"
    hy = O.Hyper.from_hparams(hp)
    gemm_mode = {"fp32": cabi.GEMM_FP32, "bf16x3": cabi.GEMM_BF16X3, "bf16": cabi.GEMM_BF16}[a.gemm]
    B, T = a.batch, T_TRAIN
    if a.strong:
        if a.batch % world:
            raise SystemExit("--strong: --batch %d is not divisible by %d GPUs" % (a.batch, world))
        B = a.batch // world
    Tp = T - hy.start_ts
    model = build_kat_model(hp)          # seeds 1234 / 7: identical replicas on every rank
    model = model.to(dev).train()
    # throughput runs keep the frame dropout of final_model.yaml active (build_kat_model disables it for parity runs)
    for name in ("p2_face", "p1_speech", "p2_speech"):
        enc = getattr(model.feature_encoder, name + "_encoder", None)
        pdrop = hp.Conditioning[name]["dropout"]
        if enc is not None and pdrop > 0:
            enc.dropout = torch.nn.Dropout(pdrop)
    model.gemm_mode = gemm_mode
    trainer = Trainer(model)
    host = make_batch(hy, B, T, seed=1 + rank, pin=True)
    dbatch = {k: v.to(dev) for k, v in host.items()}
    trainer.broadcast_parameters(0)       # replicas start identical ...
    trainer.step(dbatch)                  # ... ActNorm data-dependent init (rank 0's, broadcast inside step) + first step (untimed)
    L = cabi.lib()

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        sync()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    # ---- device-resident throughput --------------------------------------------------------------------------
    clocks = ClockSampler(local)
    if not a.ncu_step:
        clocks.start()
    for _ in range(max(a.warmup, 3)):
        trainer.step(dbatch)
    if not a.ncu_step:
        sync()
        clocks.wait_first()      # the poller is running before the timed region starts ...
        for _ in range(2):       # ... and the GPU is back under load when it does
            trainer.step(dbatch)
    if a.ncu_step:
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        trainer.step(dbatch)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return
    last = {}

    def headline_step():
        last["loss"] = trainer.step(dbatch)

    n0 = L.lfi_launch_count()
    t_w0 = time.time()
    ms = timed(headline_step, a.steps)
    t_w1 = time.time()
    launches = L.lfi_launch_count() - n0
    clk = clocks.stop((t_w0, t_w1))
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, model, trainer, last["loss"])
    frames_step = B * Tp * world
    value = frames_step * a.steps / (ms / 1e3)

    # ---- end to end: pinned host inputs -> device each step, loss read back each step ---------------------------
    # (public API: lets_face_it_b200.train.HostFeed - every step copies ITS pinned host batch to the device on a copy stream
    #  and reads ITS loss back; the copy overlaps the previous step's compute and the read-back lags one step)
    feed = HostFeed(trainer)

    def e2e_step():
        return feed.step(host)   # host -> device copy of this step's inputs + device -> host read of a step's loss

    for _ in range(2):
        e2e_step()
    feed.flush()
    ms_e2e = timed(lambda: e2e_step(), a.steps)
    feed.flush()
    e2e = frames_step * a.steps / (ms_e2e / 1e3)
    h2d = sum(v.numel() * 4 for v in host.values())

    # ---- end to end over an HBM-resident corpus (SURVEY.md section 8(f) rank 4): per step the host sends the window table entries
    #      of the batch (8 bytes per sequence) instead of the 14 MB of overlapping windows; the batch is gathered on the device
    e2e_res = None
    try:
        from lets_face_it_b200.data import ResidentWindows
        from lets_face_it_b200.train import ResidentFeed
        import random as _random

        gseg = torch.Generator().manual_seed(100 + rank)
        nseg, Lseg = 48, 600   # 28,800 frames per rank (19 MB): 25,008 stride-1 windows of 80 frames
        segs = [{"p1_face": torch.randn(Lseg, hy.C, generator=gseg), "p2_face": torch.randn(Lseg, hy.in_dim["p2_face"], generator=gseg),
                 "p1_speech": torch.randn(Lseg, hy.in_dim["p1_speech"], generator=gseg),
                 "p2_speech": torch.randn(Lseg, hy.in_dim["p2_speech"], generator=gseg)} for _ in range(nseg)]
        ds = ResidentWindows(segs, T, dev, shuffle=True, rng=_random.Random(7 + rank))
        rfeed = ResidentFeed(trainer, ds)
        cursor = [0]

        def res_step():
            i0 = cursor[0]
            cursor[0] = (i0 + B) % (len(ds) - B)
            return rfeed.step(torch.arange(i0, i0 + B))

        for _ in range(2):
            res_step()
        rfeed.flush()
        ms_res = timed(lambda: res_step(), a.steps)
        rfeed.flush()
        e2e_res = {"value": frames_step * a.steps / (ms_res / 1e3), "unit": "frames/s", "h2d_bytes_per_step": 8 * B, "d2h_bytes_per_step": 4,
                   "ms_per_step": ms_res / a.steps, "corpus_frames_per_gpu": nseg * Lseg,
                   "note": "ResidentWindows: synthetic corpus resident in HBM, the reference's stride-1 window table, batch gathered on the device"}
        del ds, rfeed, segs
    except Exception as e:  # secondary number only
        e2e_res = {"error": str(e)[:200]}

    # ---- the same step captured once as a CUDA graph and replayed (single process; SURVEY.md section 8(f) rank 2) ---------------
    graphed = None
    if world == 1:
        try:
            gs = trainer.graphed(dbatch, warmup=1)
            for _ in range(3):
                gs.step()
            sync()
            ms_g = timed(lambda: gs.step(), a.steps)
            graphed = {"value": frames_step * a.steps / (ms_g / 1e3), "unit": "frames/s", "ms_per_step": ms_g / a.steps,
                       "note": "train.GraphedStep: every launch of Trainer.step (masks, forward, backward, clip, Adam; side streams "
                               "included) replayed from one CUDA graph; learning rate and Adam bias corrections read from device memory"}
            del gs
        except Exception as e:  # secondary number only
            graphed = {"error": str(e)[:300]}

    # ---- autoregressive sampling (second half of the metric): BASELINE.json configs[3] per-GPU share -------------------
    sample = None
    if not a.no_sample:
        model.eval()
        Bs, Tg = a.sample_seqs, a.sample_frames
        hs = make_batch(hy, Bs, START_TS + Tg, seed=5 + rank)
        data = {k: v.to(dev) for k, v in hs.items()}
        data["p1_face"] = torch.zeros(Bs, START_TS, hy.C, device=dev)
        model.hparams.Infer["eps"] = 0.7
        model.inference(START_TS + min(Tg, 32), data={k: v[:, :START_TS + min(Tg, 32)] for k, v in data.items()})
        model.inference(START_TS + Tg, data=data)  # full-size warm-up: workspace allocation and first touch stay outside the timed run
        n0 = L.lfi_launch_count()
        ms_s = timed(lambda: model.inference(START_TS + Tg, data=data), 1)
        sust_s = peaks()[0]
        fps_gpu = Bs * Tg / (ms_s * 1e-3)
        sample = {"value": Bs * Tg * world / (ms_s * 1e-3), "unit": "frames/s", "sequences_per_gpu": Bs, "frames_per_sequence": Tg, "eps": 0.7,
                  "ms": ms_s, "gpu_launches": int(L.lfi_launch_count() - n0),
                  "note": "SeqGlow.inference, zero seed frames, temperature 0.7; per frame: AR window gather, two tcgen05 conditioning "
                          "GEMMs, one launch walking the 16 inverse steps, all stream-ordered with no host round trip inside the call (LFI_SAMPLE_GRAPH=1 "
                          "captures the chain as a CUDA graph per chunk: measured no gain, the chain is kernel bound); no collective",
                  # the sampler is a strictly serial chain per sequence (16 inverse steps x 750 frames): latency bound, reported as the
                  # critical path per frame next to the tensor roofline of its contractions (42.38 MFLOP per frame and sequence)
                  "roofline": {"bound": "latency", "us_per_frame": 1e3 * ms_s / Tg, "us_per_inverse_step": 1e3 * ms_s / Tg / hy.K,
                               "achieved": fps_gpu * FLOP_PER_FRAME_FWD / 1e12, "peak": sust_s, "unit": "TFLOP/s",
                               "frac": fps_gpu * FLOP_PER_FRAME_FWD / 1e12 / sust_s, "peak_source": "measured (sustained)"}}
        del data, hs
        model.train()

    out = {
        "metric": "train frames/sec", "value": value, "unit": "frames/s", "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
        "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "strong" if a.strong else "weak", "vs_baseline": None,
        "dtype": "f32" if a.gemm != "bf16" else "bf16", "data": "synthetic",
        "config": {"workload": "%s training step (fwd+NLL+bwd+clip20+Adam), B=%d sequences/GPU, T=80 (56 trained "
                               "frames/seq), frame dropout on" % ("final_model.yaml" if a.variant == "final" else
                                                                  "wide variant (K=32, H=256, %s)" % hp.Glow["rnn_type"], B),
                   "global_batch": B * world, "gemm_mode": a.gemm,
                   "l2": "per-step working set (activation stash + GEMM operands, >5 GB) far exceeds the 126 MB L2; no flush needed",
                   "parallelism": "dp%d" % world},
        "clocks": clk,
        "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / a.steps},
        "gpu_launches": int(launches),
    }
    if sample is not None:
        out["sample"] = sample
    if e2e_res is not None:
        out["e2e_resident"] = e2e_res
    if graphed is not None:
        out["graphed_step"] = graphed

    if rank == 0:
        # ---- roofline of the dominant contraction: cond_transform for all 16 steps, [B*56, 920] x [920, 8192] ---------
        sust, burst, hbm, how = peaks()
        M, N, K = B * Tp, hy.K * hy.D, 920
        A = torch.randn(M, K, device=dev)
        W = torch.randn(N, K, device=dev)
        C = torch.empty(M, N, device=dev)
        bias = torch.zeros(N, device=dev)
        ws = torch.empty(max(int(L.lfi_gemm_ws_bytes(gemm_mode, 0, 1, M, N, K, 1)), 256), dtype=torch.uint8, device=dev)

        def gemm():
            cabi.check(L.lfi_gemm(gemm_mode, 0, 1, M, N, K, A.data_ptr(), K, 0, W.data_ptr(), K, 0, C.data_ptr(), N, 0, bias.data_ptr(), 0,
                                  None, 0, 0, 1, cabi.EPI_BIAS | cabi.EPI_LRELU, ws.data_ptr(), ws.numel(), cabi.stream_ptr()), "lfi_gemm")

        for _ in range(3):
            gemm()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            gemm()
        e1.record()
        torch.cuda.synchronize()
        gms = e0.elapsed_time(e1) / 5
        ach = 2.0 * M * N * K / (gms * 1e-3) / 1e12
        traffic = None
        tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.isfile(tp):
            try:
                with open(tp) as f:
                    traffic = json.load(f).get(a.gemm, {}).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        step_traffic = None
        sp = os.path.join(ROOT, "profiles", "r02_step_traffic_default.json")
        if os.path.isfile(sp):
            try:
                with open(sp) as f:
                    st_ = json.load(f)
                step_traffic = {"dram_bytes_per_step": st_.get("step_dram_bytes"), "read": st_.get("step_dram_read"), "write": st_.get("step_dram_write"),
                                "source": "ncu dram__bytes_read/write.sum summed over every kernel of one step (scripts/gpu_r2_traffic.sh, profiles/r02_step_traffic_default.json); not re-measured in this run"}
            except Exception:
                step_traffic = None
        products = 3 if a.gemm == "bf16x3" else 1
        # canonical training FLOP per frame and sequence (SURVEY.md section 8(d)): final 127.15 M; wide (K=32, H=256) LSTM 306.6 M, GRU 267.5 M
        flop_frame = {"final": FLOP_PER_FRAME_TRAIN, "wide-lstm": 6.0 * 51102208, "wide-gru": 6.0 * 44581376}[a.variant]
        out["roofline"] = {"bound": "tensor", "achieved": ach, "peak": burst, "unit": "TFLOP/s", "frac": ach / burst, "traffic": traffic,
                           "kernel": "tc::gemm_tc_kernel, cond_transform for all 16 steps [%d x %d x %d], mode %s" % (M, N, K, a.gemm),
                           "peak_source": how + " (burst: kernel timed alone)",
                           "algorithmic_flop_per_launch": 2.0 * M * N * K, "ms_per_launch": gms,
                           "mma_products_per_flop": products, "tensor_pipe_frac": ach * products / burst,
                           "note": "achieved = algorithmic 2MNK / CUDA-event time; the split-bf16 (bf16x3) parity mode issues 3 tcgen05 "
                                   "products per algorithmic product, so tensor_pipe_frac = 3 x frac is the tensor-pipe utilisation",
                           "traffic_source": "ncu capture of this same stand-alone launch (profiles/roofline_traffic.json); not re-measured in this run",
                           "step_traffic": step_traffic,
                           "step_flop_per_frame": flop_frame,
                           "step_frac_of_tensor_roofline": value / world * flop_frame / 1e12 / sust}
        del A, W, C

        # ---- secondary: split-bf16 forward and flow core (z / NLL unchanged), single bf16 products in the backward GEMMs ---------
        if world == 1 and a.gemm == "bf16x3" and not a.no_bf16:
            try:
                os.environ["LFI_BWD_BF16"] = "1"
                for _ in range(3):
                    trainer.step(dbatch)
                ms3 = timed(lambda: trainer.step(dbatch), max(3, a.steps // 2))
                out["bf16_backward_mode"] = {"value": B * Tp * max(3, a.steps // 2) / (ms3 / 1e3), "unit": "frames/s", "ms_per_step": ms3 / max(3, a.steps // 2),
                                             "note": "LFI_BWD_BF16=1: forward and flow core as in the headline (z, NLL identical); the time-parallel backward "
                                                     "GEMMs use the hi planes only: per-tensor gradient error <= 2.8e-3 relative L2 (stated bound 5e-3); "
                                                     "an option, not the default"}
            except Exception as e:  # secondary number only
                out["bf16_backward_mode"] = {"error": str(e)[:200]}
            finally:
                os.environ.pop("LFI_BWD_BF16", None)

        # ---- secondary: the same step with plain bf16 operands (looser stated parity bound, DESIGN.md section 5) -------------
        if world == 1 and a.gemm != "bf16" and not a.no_bf16:
            try:
                model.gemm_mode = cabi.GEMM_BF16
                tr2 = Trainer(model)
                for _ in range(3):
                    tr2.step(dbatch)
                ms2 = timed(lambda: tr2.step(dbatch), max(3, a.steps // 2))
                out["bf16_mode"] = {"value": B * Tp * max(3, a.steps // 2) / (ms2 / 1e3), "unit": "frames/s", "ms_per_step": ms2 / max(3, a.steps // 2),
                                    "note": "gate/conditioning GEMMs with single bf16 products; z within 5e-3 of max|z| (measured 1e-3), NLL within 1e-4 relative"}
                del tr2
            finally:
                model.gemm_mode = gemm_mode

        # ---- CPU baseline: the oracle port on the host cores, bounded sample -------------------------------------
        if world == 1 and not a.no_cpu_baseline:
            Bc = B  # the same step as the GPU arm (B=256: ~10 s per step on 16 cores): one warm-up, then 2-3 steps
            step, frames = cpu_reference_step_fn(hp, Bc, T)
            step()
            t0 = time.perf_counter()
            n = 0
            while n < 2 or (time.perf_counter() - t0 < 20 and n < 4):
                step()
                n += 1
            dt = time.perf_counter() - t0
            out["cpu_baseline"] = {"value": frames * n / dt, "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port",
                                   "sample": "%d training steps of %d sequences x 56 frames (fwd+bwd+clip+Adam), oracle port on torch CPU fp32" % (n, Bc)}
            if sample is not None:
                # the sampling half of the metric on the host cores: oracle port, 64 sequences x 16 generated frames
                from tests.kat import build_kat_model as _bk, oracle_params_from as _op
                Pc = {k: v.detach() for k, v in _op(_bk(hp)).items()}
                Bsc, Tgc = 64, 16
                dc = O.synthetic_batch(hy, Bsc, START_TS + Tgc, seed=5)
                dc["p1_face"] = torch.zeros(Bsc, START_TS, hy.C)
                O.seq_inference(Pc, hy, dc, START_TS + 4, eps=0.7)
                t0 = time.perf_counter()
                O.seq_inference(Pc, hy, dc, START_TS + Tgc, eps=0.7)
                dts = time.perf_counter() - t0
                out["sample"]["cpu_baseline"] = {"value": Bsc * Tgc / dts, "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port",
                                                 "sample": "%d sequences x %d generated frames, oracle port on torch CPU fp32" % (Bsc, Tgc)}
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
