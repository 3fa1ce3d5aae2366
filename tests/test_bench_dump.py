"""CPU: bench.py's argument checks and the files `--dump-outputs` writes (format, size bound, fixed sample)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.helpers import ROOT


@pytest.mark.parametrize("args, message", [
    (["--steps", "0"], "--steps must be at least 1"),
    (["--impl", "reference", "--dump-outputs", "unused"], "--dump-outputs"),
    (["--ncu-step", "--dump-outputs", "unused"], "--dump-outputs"),
])
def test_bench_rejects_bad_arguments(args, message, tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=120,
                       cwd=str(tmp_path))
    assert r.returncode == 2, (r.stdout[-1000:], r.stderr[-1000:])
    assert message in r.stderr
    assert not os.path.exists(os.path.join(str(tmp_path), "unused"))


class _Trainer:
    def grad_norm(self):
        return torch.tensor(3.25)


def test_dump_outputs_writes_a_fixed_sample_of_the_parameters(tmp_path):
    import bench
    from tests.helpers import final_hparams
    from tests.kat import build_kat_model

    m = build_kat_model(final_hparams())
    flat = torch.cat([p.detach().reshape(-1) for _, p in m.named_parameters()])
    assert flat.numel() > bench.DUMP_PARAMS
    dirs = [os.path.join(str(tmp_path), d) for d in ("a", "b")]
    for d in dirs:
        bench.dump_outputs(d, m, _Trainer(), torch.tensor(-1234.5))
    got = [{n: np.load(os.path.join(d, n + ".npy")) for n in ("loss", "grad_norm", "params")} for d in dirs]
    a, b = got
    assert a["loss"].dtype == np.float64 and float(a["loss"]) == -1234.5
    assert a["grad_norm"].dtype == np.float64 and float(a["grad_norm"]) == 3.25
    assert a["params"].dtype == np.float32 and a["params"].shape == (bench.DUMP_PARAMS,)
    assert sum(os.path.getsize(os.path.join(dirs[0], f)) for f in os.listdir(dirs[0])) <= 64 << 20
    for n in a:
        assert np.array_equal(a[n], b[n]), n
    pick = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:bench.DUMP_PARAMS].sort().values
    assert np.array_equal(a["params"], flat[pick].numpy())
