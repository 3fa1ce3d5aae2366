"""Phase split of one steady-state training step with CUDA events (forward call, backward call, optimizer)."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests.helpers import final_hparams
from tests.kat import build_kat_model, kat_batch, to_device
from lets_face_it_b200 import _cabi as cabi
from lets_face_it_b200.train import Trainer
hp = final_hparams()
m = build_kat_model(hp, "cuda:0"); m.glow.set_actnorm_init(True); m.gemm_mode = cabi.GEMM_BF16X3; m.train()
batch = to_device(kat_batch(hp, 256, 80, seed=14), "cuda:0")
tr = Trainer(m)
for _ in range(4): tr.step(batch)
eng = tr.eng
ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
acc = [0.0] * 4
N = 10
for _ in range(N):
    masks = m._masks(56, 256, eng.theta.device)
    ev[0].record()
    z, nll = eng.train_forward(batch, masks)
    ev[1].record()
    tr.gflat.zero_()
    eng.train_backward(z, tr._dnll[(56, 256, 1.0)], tr.gflat)
    ev[2].record()
    tr._advance()
    tr._update(tr.gflat[:eng.n_theta], None)
    ev[3].record()
    torch.cuda.synchronize()
    for i in range(3): acc[i] += ev[i].elapsed_time(ev[i + 1])
print("forward %.3f ms | backward %.3f ms | clip+adam %.3f ms | sum %.3f" % (acc[0] / N, acc[1] / N, acc[2] / N, sum(acc[:3]) / N))
