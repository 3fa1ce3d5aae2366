"""TEST INFRASTRUCTURE ONLY — import shim for the *live* reference.

The reference is a checkout of jonepatr/lets_face_it named by the environment variable
LFI_REFERENCE_ROOT; it is not part of this repository, and without the variable the tests marked
`reference` skip.  Makes `$LFI_REFERENCE_ROOT/code/glow_pytorch/glow/{models,modules}.py` importable without editing
the reference: `glow/__init__.py:2` pulls in `glow/utils.py`, which imports `jsmin` and
`pytorch_lightning.Trainer` (utils.py:7,9); both are absent here, so two stub modules are
inserted first (SURVEY.md §8(c)).  Used by `oracle/make_golden.py` and by the
reference-only pinning tests.
"""
import argparse
import os
import sys
import types

REF_ROOT = os.environ.get("LFI_REFERENCE_ROOT", "")
REF_CODE = os.path.join(REF_ROOT, "code")
REF_YAML_DIR = os.path.join(REF_CODE, "glow_pytorch", "hparams")


def reference_available() -> bool:
    return bool(REF_ROOT) and os.path.isfile(os.path.join(REF_CODE, "glow_pytorch", "glow", "models.py"))


def import_reference():
    """Returns (models, modules) of the unmodified reference."""
    if not reference_available():
        raise RuntimeError("reference tree not found: set LFI_REFERENCE_ROOT to a checkout of jonepatr/lets_face_it (now %r)" % REF_ROOT)
    if "jsmin" not in sys.modules:
        m = types.ModuleType("jsmin")
        m.jsmin = lambda s: s
        sys.modules["jsmin"] = m
    if "pytorch_lightning" not in sys.modules:
        pl = types.ModuleType("pytorch_lightning")

        class Trainer:  # only add_argparse_args is touched at import time
            @staticmethod
            def add_argparse_args(p):
                return p

        pl.Trainer = Trainer
        pl.LightningModule = object
        sys.modules["pytorch_lightning"] = pl
    if REF_CODE not in sys.path:
        sys.path.insert(0, REF_CODE)
    from glow_pytorch.glow import models, modules  # noqa: E402

    return models, modules


def load_reference_hparams(name="final_model.yaml"):
    import yaml

    with open(os.path.join(REF_YAML_DIR, name)) as f:
        return argparse.Namespace(**yaml.safe_load(f))
