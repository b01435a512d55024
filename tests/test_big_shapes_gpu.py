"""GPU parity at the BENCHMARKED shapes (BASELINE.json configs 2-4): SPADEGenerator 1024x768 batch 8, ConditionGenerator 1024x768
batch 4 — buffers beyond 2^31 bytes, 6144 pixel tiles per image, `long long` pixel offsets — against goldens of the UNMODIFIED
reference (tests/golden/gen_1024x768_b8.npz / tocg_1024x768_b4.npz: stride-8 sub-sampling of every output, full-resolution crops
at the image corners/centre, per-image per-channel sums; written by tests/golden/make_golden.py --only big).  Bounds: 1.1 x the
storage-rounded oracle's own deviation, measured on image 0 at full size (tests/floors.py model)."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "oracle"))
import hrviton_oracle as orc  # noqa: E402
import floors  # noqa: E402
from helpers import gen_opt, load_golden, pick, synth_state_dict, tocg_opt  # noqa: E402
from hrviton_b200 import ops, synth  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(params=["bf16", "fp16"])
def precision(request):
    ops.set_precision(request.param)
    yield request.param
    ops.set_precision("bf16")


def _gen_floor_image0(g, sd, x, seg, seed, n, precision):
    """Rounded-oracle deviation on image 0 of the batch (full 1024x768), against the golden's sub-sampling of that image."""
    cnt = [0]

    def noise(b, hh, ww):
        t = synth.spade_noise(n, hh, ww, seed, cnt[0])[0:1]
        cnt[0] += 1
        return t

    with torch.no_grad(), orc.storage_rounding(floors.DT[precision]):
        out = orc.spade_generator_forward(sd, x[0:1], seg[0:1], noise)
    crops = torch.stack([out[:, :, y:y + 64, x0:x0 + 64] for y, x0 in g["crop_yx"]], 1)
    return (floors.stats(pick(g, "sub8", out[:, :, ::8, ::8]), g["sub8"][0:1].astype(np.float32)),
            floors.stats(pick(g, "crops", crops), g["crops"][0:1].astype(np.float32)))


def test_generator_1024x768_b8(precision):
    import network_generator
    g = load_golden("gen_1024x768_b8")
    n, h, w = [int(v) for v in g["shape"]]
    seed = int(g["seed"])
    sd = synth_state_dict("gen", seed)
    m = network_generator.SPADEGenerator(gen_opt(h, w, True), 9)
    m.load_state_dict(sd)
    m = m.cuda().eval()
    cnt = [0]

    def noise(b, hh, ww):
        t = synth.spade_noise(b, hh, ww, seed, cnt[0]).cuda()
        cnt[0] += 1
        return t

    m.noise_source = noise
    x, seg = synth.gen_inputs(n, h, w, seed)
    with torch.no_grad():
        out = m(x.cuda(), seg.cuda())
    torch.cuda.synchronize()
    assert out.shape == (n, 3, h, w) and bool(torch.isfinite(out).all())
    fl, fl_crops = _gen_floor_image0(g, sd, x, seg, seed, n, precision)
    outc = out.cpu()
    sub8 = pick(g, "sub8", outc[:, :, ::8, ::8])
    crops = pick(g, "crops", torch.stack([outc[:, :, y:y + 64, x0:x0 + 64] for y, x0 in g["crop_yx"]], 1))
    smax = s2max = 0.0
    for i in range(n):  # per image against the image-0 floor: same sample count on both sides of every ratio
        s = floors.check("%s gen 1024x768 img%d sub8" % (precision, i), sub8[i:i + 1], g["sub8"][i:i + 1].astype(np.float32), fl)
        s2 = floors.check("%s gen 1024x768 img%d crops" % (precision, i), crops[i:i + 1], g["crops"][i:i + 1].astype(np.float32), fl_crops)
        smax, s2max = max(smax, s["max"]), max(s2max, s2["max"])
    dmean = np.abs(outc.double().sum((2, 3)).numpy() - g["chan_sums"]) / float(h * w)
    print("PARITY %s gen 1024x768 per-image channel-mean error max %.3e (floor mean|d| %.3e)" % (precision, dmean.max(), fl["mean"]))
    assert dmean.max() <= fl["mean"]  # the signed mean error of a whole 786k-pixel plane sits far below the mean |error|
    if precision == "fp16":
        assert smax < 1e-2 and s2max < 1e-2  # north-star tolerance as written, at the benchmarked shape, every image


def test_tocg_1024x768_b4(precision):
    import networks
    g = load_golden("tocg_1024x768_b4")
    n, h, w = [int(v) for v in g["shape"]]
    seed = int(g["seed"])
    sd = synth_state_dict("tocg", seed)
    m = networks.ConditionGenerator(tocg_opt(True), 4, 16, 13, ngf=96, norm_layer=torch.nn.BatchNorm2d)
    m.load_state_dict(sd)
    m = m.cuda().eval()
    i1, i2 = synth.tocg_inputs(n, h, w, seed)
    with torch.no_grad():
        flows, seg, wc, wcm = m(i1.cuda(), i2.cuda())
    torch.cuda.synchronize()
    with torch.no_grad(), orc.storage_rounding(floors.DT[precision]):  # the rounded oracle on the same 4 images
        rf, rs, rwc, rwcm = orc.tocg_forward(sd, i1, i2)
    step = lambda i: 1 if i < 3 else 4
    segc, wcc, wcmc = seg.cpu(), wc.cpu(), wcm.cpu()
    items = [("seg_sub8", segc[:, :, ::8, ::8], rs[:, :, ::8, ::8], 0.0), ("seg_crop", segc[:, :, h - 64:, w - 64:], rs[:, :, h - 64:, w - 64:], 0.0),
             ("warped_c_sub8", wcc[:, :, ::8, ::8], rwc[:, :, ::8, ::8], 0.0), ("warped_cm_sub8", wcmc[:, :, ::8, ::8], rwcm[:, :, ::8, ::8], 5e-3)]
    for i, f in enumerate(flows):
        items.append(("flow%d_sub" % i, f.cpu()[:, ::step(i), ::step(i)], rf[i][:, ::step(i), ::step(i)], 0.0))
    for key, got, flo, extra in items:
        got, flo = pick(g, key, got), pick(g, key, flo)
        for i in range(n):  # image by image: local content (e.g. the 64x64 crop) sets the local error level
            fl = floors.stats(flo[i:i + 1], g[key][i:i + 1])
            s = floors.check("%s tocg 1024x768 img%d %s" % (precision, i, key), got[i:i + 1], g[key][i:i + 1], fl, extra_abs=extra)
            if precision == "fp16" and not key.startswith("flow"):
                assert s["max"] < 1e-2 * max(1.0, s["absmax"]), (key, s)
    # whole-plane signed mean error per (image, channel) against the same quantity of the rounded oracle (image 0)
    dmean = np.abs(segc.double().sum((2, 3)).numpy() - g["seg_sums"]) / float(h * w)
    dmean_floor = np.abs(rs.double().sum((2, 3)).numpy() - g["seg_sums"]) / float(h * w)
    print("PARITY %s tocg 1024x768 per-plane mean error max %.3e (rounded oracle %.3e)" % (precision, dmean.max(), dmean_floor.max()))
    assert dmean.max() <= 2.0 * dmean_floor.max() + 1e-5
