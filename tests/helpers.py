"""Shared test helpers: build reference-shaped state_dicts WITHOUT the reference (the GPU box
has no /root/reference) by instantiating this repo's drop-in modules, whose state_dict keys and
shapes are identical to the reference's (tests/test_boundary.py pins that against the key lists
recorded from the live reference in tests/golden/state_keys.json)."""
import json
import os
import types

import numpy as np
import torch

from hrviton_b200 import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    d = np.load(os.path.join(GOLDEN, name + ".npz"))
    return {k: d[k] for k in d.files}


def pick(g, key, t):
    """`t` (leading dim = batch) at the positions golden `key` holds: all of them, or, where the fixture keeps a per-image sample of a
    large output, the flat per-image indices stored beside it as `<key>_idx` (make_golden.sample_large)."""
    idx = g.get(key + "_idx")
    if idx is None:
        return t
    if torch.is_tensor(t):
        t = t.detach().float().cpu()
        return t.reshape(t.shape[0], -1)[:, torch.from_numpy(idx.astype(np.int64))]
    t = np.asarray(t)
    return t.reshape(t.shape[0], -1)[:, idx]


def state_shapes(kind):
    with open(os.path.join(GOLDEN, "state_keys.json")) as f:
        return json.load(f)[kind]


def synth_state_dict(kind, seed):
    """Reference-shaped state_dict filled by synth.fill_state_dict — identical to what
    make_golden.py loaded into the reference module."""
    sd = {}
    for k, (shape, dtype) in state_shapes(kind).items():
        sd[k] = torch.zeros(shape, dtype=getattr(torch, dtype))
    synth.fill_state_dict(sd, seed)
    return sd


def tocg_opt(cuda=False):
    return types.SimpleNamespace(warp_feature="T1", out_layer="relu", cuda=cuda)


def gen_opt(h, w, cuda=False):
    return types.SimpleNamespace(norm_G="spectralaliasinstance", gen_semantic_nc=7, ngf=64,
                                 num_upsampling_layers="most", fine_height=h, fine_width=w, cuda=cuda,
                                 ndf=64, norm_D="spectralinstance", n_layers_D=3, num_D=2, no_ganFeat_loss=False,
                                 init_type="xavier", init_variance=0.02)


def maxdiff(a, b):
    a = a.detach().float().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    b = b.detach().float().cpu().numpy() if torch.is_tensor(b) else np.asarray(b)
    assert a.shape == b.shape, (a.shape, b.shape)
    return float(np.abs(a - b).max())
