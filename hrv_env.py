"""Environment for running the reference scripts unchanged against this repository's drop-in modules (see shims/README.md).

    import hrv_env; hrv_env.install()          # repo root first on sys.path, shims/ last, numpy aliases restored
    hrv_env.load_reference_script("train_generator")   # imports the original train_generator (reference_dir()) with
                                                        # `networks`, `network_generator`, `sync_batchnorm` bound to the drop-ins
"""
import importlib.util
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
SHIMS = os.path.join(ROOT, "shims")


def install():
    import numpy as np
    for name, typ in (("float", float), ("int", int), ("bool", bool)):
        if not hasattr(np, name):
            setattr(np, name, typ)
    import torch
    if not getattr(torch.optim.Adam, "_hrv_betas_patch", False):
        # train_generator.py:154,157 passes betas=(0, 0.9): an int next to a float, which torch >= 2.6 rejects ("betas must be either
        # both floats or both Tensors") — an incompatibility between the 2022 script and today's torch, not with this repository
        _init = torch.optim.Adam.__init__

        def _adam_init(self, params, lr=1e-3, betas=(0.9, 0.999), *a, **k):
            betas = tuple(b if torch.is_tensor(b) else float(b) for b in betas)
            return _init(self, params, lr, betas, *a, **k)

        torch.optim.Adam.__init__ = _adam_init
        torch.optim.Adam._hrv_betas_patch = True
    if ROOT in sys.path:
        sys.path.remove(ROOT)
    sys.path.insert(0, ROOT)
    if SHIMS not in sys.path:
        sys.path.append(SHIMS)  # last: a real torchgeometry / tensorboardX / apex wins
    os.environ.setdefault("HRV_VGG_RANDOM_INIT", "1" if not os.path.exists(os.path.expanduser("~/.cache/torch/hub/checkpoints/vgg19-dcbb9e9d.pth")) else "0")


def reference_dir():
    """Where the original HR-VITON modules are: the checkout named by $HRV_REFERENCE_DIR, else the compiled modules that
    __graft_entry__.build() placed in oracle/_ref (oracle/build_reference.py), else None.  This repository does not ship them."""
    for d in (os.environ.get("HRV_REFERENCE_DIR"), os.path.join(ROOT, "oracle", "_ref")):
        if d and reference_file(d, "train_generator"):
            return d
    return None


def reference_file(d, name):
    """<d>/<name>.py of a checkout, or the sourceless <d>/<name>.pyc of a compiled one; None when neither exists."""
    for f in (name + ".py", name + ".pyc"):
        if os.path.isfile(os.path.join(d, f)):
            return os.path.join(d, f)
    return None


def load_reference_script(name, alias=None):
    """Imports <reference>/<name>.py as a module.  Its own sibling imports that this repo replaces (networks, network_generator,
    sync_batchnorm) resolve to the drop-ins at the repo root; the rest (utils, cp_dataset, eval_models) to the reference's files."""
    install()
    d = reference_dir()
    if d is None:
        raise FileNotFoundError("no reference modules: build with a checkout of the original HR-VITON repository, or set HRV_REFERENCE_DIR")
    import network_generator  # noqa: F401  (bind the drop-ins before the reference directory becomes importable)
    import networks  # noqa: F401
    import sync_batchnorm  # noqa: F401
    if d not in sys.path:
        sys.path.insert(1, d)  # after the repo root
    spec = importlib.util.spec_from_file_location(alias or ("ref_" + name), reference_file(d, name))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod
