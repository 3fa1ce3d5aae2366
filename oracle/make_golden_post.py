"""TEST INFRASTRUCTURE ONLY — golden vectors for the rows of SURVEY.md §8(f) ranks 2-3 (output wire format of sampling,
training-step glue), produced by the UNMODIFIED reference (a jonepatr/lets_face_it checkout):

    LFI_REFERENCE_ROOT=<checkout> python oracle/make_golden_post.py    # writes tests/golden/kat_post.npz

* `expand_face_dim` is executed from the reference's own source text (`code/glow_pytorch/generate_motion_from_model.py`:
  the module itself imports rendering / Lightning / optuna packages that are absent here, so only that function's `def`
  block is compiled, unmodified, with `torch` in scope), followed by the de-standardisation of `generate_motion` (:68).
* `derange_batch` and `get_mismatched_modalities` are imported from `glow_pytorch.glow.utils` through the shim.
"""
import ast
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle.ref_shim import REF_CODE, import_reference, load_reference_hparams  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def reference_function(path, name):
    src = open(path).read()
    for node in ast.parse(src).body:
        if isinstance(node, ast.FunctionDef) and node.name == name:
            ns = {"torch": torch}
            exec(compile(ast.Module(body=[node], type_ignores=[]), path, "exec"), ns)
            return ns[name]
    raise KeyError(name)


def main():
    import_reference()
    from glow_pytorch.glow.utils import calc_jerk, derange_batch, get_mismatched_modalities

    hp = load_reference_hparams()
    expand = reference_function(os.path.join(REF_CODE, "glow_pytorch", "generate_motion_from_model.py"), "expand_face_dim")
    g = torch.Generator().manual_seed(3)
    seq = torch.randn(3, 7, 56, generator=g)
    means = torch.randn(56, generator=g)
    stds = torch.rand(56, generator=g) + 0.5
    out = {"seq": seq.numpy(), "means": means.numpy(), "stds": stds.numpy(),
           "expanded": expand(seq, hp.Data).numpy(),
           "destd_expanded": expand(seq * stds + means, hp.Data).numpy(),   # generate_motion_from_model.py:68-70
           "data_dims": np.array([hp.Data["expression_dim"], hp.Data["jaw_dim"], hp.Data["neck_dim"]])}
    batch = {"p1_face": torch.randn(6, 4, 5, generator=g), "p2_face": torch.randn(6, 4, 5, generator=g),
             "p1_speech": torch.randn(6, 4, 3, generator=g), "p2_speech": torch.randn(6, 4, 3, generator=g)}
    mods, name = get_mismatched_modalities(hp)
    torch.manual_seed(99)
    mixed = derange_batch(batch, mods)
    for k, v in batch.items():
        out["batch_" + k] = v.numpy()
        out["deranged_" + k] = mixed[k].numpy()
    # validation metric of mimicry_logger.py:175-184: calc_jerk (glow/utils.py:53-58) on seeded frames
    jx = torch.randn(5, 40, 56, generator=g) * 0.7
    out["jerk_x"] = jx.numpy()
    out["jerk"] = np.float32(calc_jerk(jx))
    out["mismatched_modalities"] = np.array(mods)
    out["mismatched_name"] = np.array(name)
    np.savez_compressed(os.path.join(GOLDEN, "kat_post.npz"), **out)
    print("wrote kat_post.npz:", {k: getattr(v, "shape", None) for k, v in out.items()})


if __name__ == "__main__":
    main()
