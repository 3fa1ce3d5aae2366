"""Known-answer-test recipe of SURVEY.md §8(c), applied to THIS package's drop-in modules (the constructor
draws from the torch / numpy RNG streams exactly as the reference does, so seeds give identical parameters)."""
import numpy as np
import torch

from oracle import glow_oracle as O


def build_kat_model(hp, device=None):
    from lets_face_it_b200.glow import LinearZeros, ModalityEncoder, SeqGlow

    torch.manual_seed(1234)
    np.random.seed(1234)
    m = SeqGlow(hp)
    g = torch.Generator().manual_seed(7)
    for mod in m.modules():
        if isinstance(mod, LinearZeros):
            with torch.no_grad():
                mod.weight.copy_(torch.randn(mod.weight.shape, generator=g) * 0.05)
                mod.bias.copy_(torch.randn(mod.bias.shape, generator=g) * 0.05)
                mod.logs.copy_(torch.randn(mod.logs.shape, generator=g) * 0.1)
    for mod in m.modules():
        if isinstance(mod, ModalityEncoder):
            mod.dropout = None
    if device is not None:
        m = m.to(device)
    return m


# torch splits a large CPU reduction into one partial sum per intra-op thread, so the last bits of a double-precision sum
# depend on the thread count: the stored fingerprints (tests/golden/kat_*.npz) were summed with 8 threads, and summing
# with 16 threads moves them by ~2e-12.  Pinning the count is necessary, not sufficient: the order also follows the vector
# width of the CPU kernel torch dispatches to (the same results were seen under AVX2 and AVX-512, not on other ISAs), and
# OpenMP must grant all 8 threads (OMP_THREAD_LIMIT, OMP_DYNAMIC).  The parameters themselves are bit-identical, so a
# host where the sums still differ needs a comparison within a few ulp, not a looser parameter check.
FINGERPRINT_THREADS = 8


def fingerprint(sd):
    names = sorted(sd.keys())
    threads = torch.get_num_threads()
    torch.set_num_threads(FINGERPRINT_THREADS)
    try:
        return names, np.array([[float(sd[n].double().sum()), float(sd[n].double().abs().sum())] for n in names])
    finally:
        torch.set_num_threads(threads)


def to_device(batch, device):
    return {k: v.to(device) for k, v in batch.items()}


def oracle_params_from(model):
    return {k: v.detach().cpu().float().clone() for k, v in model.state_dict().items()}


def kat_batch(hp, B, T, seed=1):
    return O.synthetic_batch(O.Hyper.from_hparams(hp), B, T, seed)
