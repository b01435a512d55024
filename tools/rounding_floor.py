"""CPU experiment behind DESIGN.md "Parity": how far does the fp32 oracle itself move when its convolutions round their
inputs / weights / outputs to bf16 or fp16 (oracle.storage_rounding)?  Prints max / mean |delta| per output against the
committed reference goldens.  python tools/rounding_floor.py [gen|tocg] ..."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import hrv_loader  # noqa: E402

hrv_loader.load()
import hrviton_oracle as orc  # noqa: E402
from helpers import load_golden, pick, synth_state_dict  # noqa: E402
from hrviton_b200 import synth  # noqa: E402


def gen(name):
    g = load_golden(name)
    n, h, w = [int(v) for v in g["shape"]]
    seed = int(g["seed"])
    sd = synth_state_dict("gen", seed)
    x, seg = synth.gen_inputs(n, h, w, seed)
    for dt, outs in ((None, True), (torch.bfloat16, True), (torch.bfloat16, False), (torch.float16, True)):
        cnt = [0]

        def noise(b, hh, ww):
            t = synth.spade_noise(b, hh, ww, seed, cnt[0])
            cnt[0] += 1
            return t
        with torch.no_grad(), orc.storage_rounding(dt, outs):
            out = orc.spade_generator_forward(sd, x, seg, noise)
        d = (pick(g, "out", out).numpy() - g["out"]).__abs__()
        print("%s rounding=%s outputs=%s: max %.3e mean %.3e p99.9 %.3e" % (name, dt, outs, d.max(), d.mean(), np.quantile(d, 0.999)))


def tocg(name):
    g = load_golden(name)
    n, h, w = [int(v) for v in g["shape"]]
    seed = int(g["seed"])
    sd = synth_state_dict("tocg", seed)
    i1, i2 = synth.tocg_inputs(n, h, w, seed)
    for dt, outs in ((None, True), (torch.bfloat16, True), (torch.bfloat16, False), (torch.float16, True)):
        with torch.no_grad(), orc.storage_rounding(dt, outs):
            flows, seg, wc, wcm = orc.tocg_forward(sd, i1, i2)
        rows = [(k, pick(g, k, t), g[k]) for k, t in [("seg", seg), ("warped_c", wc), ("warped_cm", wcm)] + [("flow%d" % i, f) for i, f in enumerate(flows)]]
        print("%s rounding=%s outputs=%s: " % (name, dt, outs) + "  ".join("%s max %.2e mean %.2e" % (k, np.abs(a.numpy() - b).max(), np.abs(a.numpy() - b).mean()) for k, a, b in rows))


if __name__ == "__main__":
    torch.set_num_threads(min(16, os.cpu_count() or 1))
    what = sys.argv[1:] or ["tocg", "gen"]
    if "tocg" in what:
        tocg("tocg_256x192_b1")
    if "gen" in what:
        gen("gen_512x384_b1")
