"""CPU: the oracle restatement (oracle/hrviton_oracle.py) against fixtures produced by the live
reference modules (tests/golden/make_golden.py).  This is what pins the oracle."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "oracle"))
import hrviton_oracle as orc  # noqa: E402
from helpers import load_golden, maxdiff, pick, synth_state_dict  # noqa: E402
from hrviton_b200 import synth  # noqa: E402

TOL = 2e-5  # fp32 vs fp32, different op association only


@pytest.mark.parametrize("name", ["tocg_256x192_b1", "tocg_128x96_b2"])
def test_tocg(name):
    g = load_golden(name)
    n, h, w = [int(v) for v in g["shape"]]
    sd = synth_state_dict("tocg", int(g["seed"]))
    i1, i2 = synth.tocg_inputs(n, h, w, int(g["seed"]))
    with torch.no_grad():
        flows, seg, wc, wcm = orc.tocg_forward(sd, i1, i2)
    for i, f in enumerate(flows):
        assert maxdiff(pick(g, "flow%d" % i, f), g["flow%d" % i]) < 1e-4
    assert maxdiff(pick(g, "seg", seg), g["seg"]) < 1e-4
    assert maxdiff(pick(g, "warped_c", wc), g["warped_c"]) < 1e-4
    assert maxdiff(pick(g, "warped_cm", wcm), g["warped_cm"]) < 1e-4


@pytest.mark.parametrize("name", ["gen_512x384_b1", "gen_256x256_b2"])
def test_gen(name):
    g = load_golden(name)
    n, h, w = [int(v) for v in g["shape"]]
    seed = int(g["seed"])
    sd = synth_state_dict("gen", seed)
    x, seg = synth.gen_inputs(n, h, w, seed)
    cnt = [0]

    def noise_fn(b, hh, ww):
        t = synth.spade_noise(b, hh, ww, seed, cnt[0])
        cnt[0] += 1
        return t

    with torch.no_grad():
        out = orc.spade_generator_forward(sd, x, seg, noise_fn)
    assert cnt[0] == int(g["n_noise"]) == 23
    assert maxdiff(pick(g, "out", out), g["out"].astype(np.float32)) < 1e-3  # fixture stored as fp16


def test_gend():
    g = load_golden("gend_128x96_b2")
    n, h, w = [int(v) for v in g["shape"]]
    seed = int(g["seed"])
    sd = synth_state_dict("gend", seed)
    x, seg = synth.gen_inputs(n, h, w, seed, input_nc=3)
    with torch.no_grad():
        res = orc.gen_d_forward(sd, torch.cat([seg, x], 1))
    for i, fs in enumerate(res):
        for j, f in enumerate(fs):
            assert maxdiff(pick(g, "d%d_f%d" % (i, j), f), g["d%d_f%d" % (i, j)]) < 1e-4


def test_tocgd():
    g = load_golden("tocgd_256x192_b1")
    seed = int(g["seed"])
    sd = synth_state_dict("tocgd", seed)
    i1, i2 = synth.tocg_inputs(1, 256, 192, seed)
    segs = synth.one_hot(synth.labels((1, 256, 192), 13, seed, "dseg"), 13)
    with torch.no_grad():
        res = orc.tocg_d_forward(sd, torch.cat([i1, i2, segs], 1))
    for i, r in enumerate(res):
        assert maxdiff(r[0], g["d%d" % i]) < 1e-4


# ---- numpy index-arithmetic primitives vs the torch substrate --------------------------------

def test_np_bilinear_up2():
    x = synth.uniform((2, 3, 5, 7), 1, "u")
    ref = F.interpolate(x, scale_factor=2, mode="bilinear", align_corners=False)
    assert maxdiff(orc.np_bilinear_up2(x.numpy()), ref) < 1e-6


def test_np_nearest_and_pool():
    x = synth.uniform((1, 2, 16, 12), 2, "n")
    for oh, ow in [(8, 6), (32, 24), (2, 1), (4, 3)]:
        ref = F.interpolate(x, size=(oh, ow), mode="nearest")
        assert maxdiff(orc.np_nearest_resize(x.numpy(), oh, ow), ref) == 0.0
    for hh, ww in [(16, 12), (17, 13), (9, 7)]:
        y = synth.uniform((1, 2, hh, ww), 3, "p%d" % hh)
        ref = F.avg_pool2d(y, 3, stride=2, padding=1, count_include_pad=False)
        assert maxdiff(orc.np_avgpool3s2(y.numpy()), ref) < 1e-6


def test_np_instance_norm():
    x = synth.normalish((2, 5, 9, 7), 4, "in", 2.0, 0.5)
    ref = F.instance_norm(x, eps=1e-5)
    out, m, r = orc.np_instance_norm(x.numpy())
    assert maxdiff(out, ref) < 1e-5


def test_np_flow_warp_bit_exact_indices():
    """Warp coordinate chain: numpy fp32 restatement vs torch (upsample+div+grid+grid_sample).
    Values within 1e-6 and — the bit-exact requirement — identical integer gather indices,
    checked by warping index-ramp images."""
    n, h, w = 2, 32, 24
    flow = synth.normalish((n, h // 2, w // 2, 2), 5, "fl", 3.0)
    src = synth.uniform((n, 4, h, w), 5, "src")
    ref = orc.flow_warp(src, flow)
    x0, y0, tx, ty = orc.np_flow_warp_coords(flow.numpy(), h, w, h, w)
    out = orc.np_gather_bilinear(src.numpy(), x0, y0, tx, ty)
    assert maxdiff(out, ref) < 1e-5
    # indices: torch's own floor() of its own coordinates, reproduced through torch ops
    fl = F.interpolate(flow.permute(0, 3, 1, 2), scale_factor=2, mode="bilinear", align_corners=False)
    gx = fl[:, 0] / ((w / 2 - 1.0) / 2.0) + torch.linspace(-1, 1, w)[None, None, :]
    gy = fl[:, 1] / ((h / 2 - 1.0) / 2.0) + torch.linspace(-1, 1, h)[None, :, None]
    ix = (((gx + 1) * w - 1) / 2).clamp(0, w - 1)
    iy = (((gy + 1) * h - 1) / 2).clamp(0, h - 1)
    assert np.array_equal(ix.floor().int().numpy(), x0)
    assert np.array_equal(iy.floor().int().numpy(), y0)
    # lerp weights agree to an ulp of the coordinate (torch may contract to FMA; numpy does not)
    assert np.abs((ix - ix.floor()).numpy() - tx).max() < 4e-6


def test_np_spectral_sigma():
    sd = synth_state_dict("gen", 23)
    p = "up_3.conv_0"
    s = orc.np_spectral_sigma(sd[p + ".weight_orig"].numpy(), sd[p + ".weight_u"].numpy(), sd[p + ".weight_v"].numpy())
    w = orc.spectral_weight(sd, p)
    assert abs(float((sd[p + ".weight_orig"] / w).flatten()[0]) - s) < 1e-4 * abs(s)


def test_storage_rounding_floor_model():
    """The storage-rounding model behind the GPU parity bounds (tests/floors.py): rounding the oracle's convolutions to bf16 moves
    its own output beyond the 1e-2 north-star tolerance (so no bf16-storage implementation can meet it in max-norm), rounding to
    fp16 stays inside it, and no rounding reproduces the golden."""
    import floors
    bf = floors.gen_floor("gen_256x256_b2", "bf16")["out"]
    hf = floors.gen_floor("gen_256x256_b2", "fp16")["out"]
    print("floor gen_256x256_b2: bf16 max %.3e mean %.3e | fp16 max %.3e mean %.3e" % (bf["max"], bf["mean"], hf["max"], hf["mean"]))
    assert bf["max"] > 1e-2 and hf["max"] < 1e-2 and hf["mean"] < bf["mean"] / 4
    t = floors.tocg_floor("tocg_128x96_b2", "fp16")
    assert max(v["max"] for v in t.values()) < 1e-2
