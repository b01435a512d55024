"""Storage-rounding floors: what 16-bit activation storage costs the fp32 algorithm ITSELF.

The CPU oracle is re-run with every convolution rounding its input activations, weights and output to bf16 / fp16
(oracle.storage_rounding; gradients are rounded at the same points on the way back) and compared with the fp32 goldens of the
unmodified reference.  The GPU parity tests then require the CUDA kernels to deviate from the same goldens by no more than
RATIO x that floor, statistic by statistic — the bound is derived, not hand-picked.  Results are cached per session."""
import functools
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "oracle"))
import hrviton_oracle as orc  # noqa: E402
from helpers import load_golden, pick, synth_state_dict  # noqa: E402
from hrviton_b200 import synth  # noqa: E402

RATIO = 1.1          # kernels may deviate by at most this factor times the rounded oracle's own deviation (mean, tail quantile)
# max|delta| is ONE sample from the tail of the error distribution, so it moves between equally valid realisations of the same rounding
# noise while mean and tail quantile do not.  Measured in round 2: the one-CTA and the CTA-pair convolution kernels produce the same
# products in a different fp32 summation order; on tocg_128x96 warped_c the max went 1.3x -> 1.57x the floor's max between them with the
# mean at 1.09x and the 99.9 % quantile at 1.11x in both.  The bound below covers that spread; a real defect moves mean and tail too.
RATIO_MAX = 1.6
DT = {"bf16": torch.bfloat16, "fp16": torch.float16}
# The floor is ONE realisation of the rounding noise and the kernels' error is another (different rounding points inside fused
# epilogues, different accumulation order), so a ratio of two sample statistics carries sampling noise of its own.  The bounds are
# therefore RATIO x floor x (1 + 2/sqrt(n_eff)): n_eff = n/16 for the mean (errors are spatially correlated over ~16 samples), the
# number of samples beyond the quantile for the tail statistic and the maximum.  For the large outputs that matter (>= 1e5 samples)
# the allowance is below 2% (mean) and the bound is the plain 1.1x; it only widens for tiny tensors (a 8x6x2 flow has 96 samples).


def _tail_q(n):
    """Tail quantile with at least 64 samples beyond it (p99.9 from 64k samples up; None below 640 samples: only mean/max)."""
    if n < 640:
        return None
    return 1.0 - max(64.0, n / 1000.0) / n


def stats(got, ref):
    got = got.detach().float().cpu().numpy() if torch.is_tensor(got) else np.asarray(got, np.float32)
    ref = ref.detach().float().cpu().numpy() if torch.is_tensor(ref) else np.asarray(ref, np.float32)
    assert got.shape == ref.shape, (got.shape, ref.shape)
    d = np.abs(got - ref).ravel()
    q = _tail_q(d.size)
    return {"max": float(d.max()), "mean": float(d.mean()), "tail": float(np.quantile(d, q)) if q is not None else None, "q": q,
            "n": int(d.size), "absmax": float(np.abs(ref).max())}


def check(name, got, ref, floor, log=print, extra_abs=0.0):
    """Assert stats(got, ref) <= RATIO * floor * (1 + sampling allowance), statistic by statistic; prints the measured ratios.
    `floor` must come from a tensor of the same shape (same sample count) as got/ref."""
    s = stats(got, ref)
    assert s["n"] == floor["n"], (name, s["n"], floor["n"])
    n = s["n"]
    tail_n = n * (1.0 - s["q"]) if s["q"] is not None else float(n)
    a_mean, a_tail = 1.0 + 2.0 / np.sqrt(max(n / 16.0, 1.0)), 1.0 + 2.0 / np.sqrt(tail_n)
    r = {k: (s[k] / max(floor[k], 1e-12) if s[k] is not None else float("nan")) for k in ("max", "mean", "tail")}
    log("PARITY %-34s n=%-8d max %.3e (floor %.3e, x%.2f <= %.2f)  mean %.3e (floor %.3e, x%.2f <= %.2f)  tail[q=%s] x%.2f <= %.2f  ref absmax %.3g"
        % (name, n, s["max"], floor["max"], r["max"], RATIO_MAX * a_tail, s["mean"], floor["mean"], r["mean"], RATIO * a_mean,
           ("%.4f" % s["q"]) if s["q"] is not None else "-", r["tail"], RATIO * a_tail, s["absmax"]))
    assert s["mean"] <= RATIO * a_mean * floor["mean"] + extra_abs, (name, "mean", s["mean"], floor["mean"])
    if s["q"] is not None:
        assert s["tail"] <= RATIO * a_tail * floor["tail"] + extra_abs, (name, "tail", s["tail"], floor["tail"])
    assert s["max"] <= RATIO_MAX * a_tail * floor["max"] + extra_abs, (name, "max", s["max"], floor["max"])
    return s


@functools.lru_cache(maxsize=None)
def tocg_floor(name, precision):
    g = load_golden(name)
    n, h, w = [int(v) for v in g["shape"]]
    seed = int(g["seed"])
    sd = synth_state_dict("tocg", seed)
    i1, i2 = synth.tocg_inputs(n, h, w, seed)
    with torch.no_grad(), orc.storage_rounding(DT[precision]):
        flows, seg, wc, wcm = orc.tocg_forward(sd, i1, i2)
    out = {"seg": stats(pick(g, "seg", seg), g["seg"]), "warped_c": stats(pick(g, "warped_c", wc), g["warped_c"]),
           "warped_cm": stats(pick(g, "warped_cm", wcm), g["warped_cm"])}
    for i, f in enumerate(flows):
        out["flow%d" % i] = stats(pick(g, "flow%d" % i, f), g["flow%d" % i])
    return out


@functools.lru_cache(maxsize=None)
def gen_floor(name, precision):
    g = load_golden(name)
    n, h, w = [int(v) for v in g["shape"]]
    seed = int(g["seed"])
    sd = synth_state_dict("gen", seed)
    x, seg = synth.gen_inputs(n, h, w, seed)
    cnt = [0]

    def noise(b, hh, ww):
        t = synth.spade_noise(b, hh, ww, seed, cnt[0])
        cnt[0] += 1
        return t

    with torch.no_grad(), orc.storage_rounding(DT[precision]):
        out = orc.spade_generator_forward(sd, x, seg, noise)
    return {"out": stats(pick(g, "out", out), g["out"])}


@functools.lru_cache(maxsize=None)
def gend_floor(name, precision):
    g = load_golden(name)
    n, h, w = [int(v) for v in g["shape"]]
    seed = int(g["seed"])
    sd = synth_state_dict("gend", seed)
    x, seg = synth.gen_inputs(n, h, w, seed, input_nc=3)
    with torch.no_grad(), orc.storage_rounding(DT[precision]):
        res = orc.gen_d_forward(sd, torch.cat([seg, x], 1))
    return {"d%d_f%d" % (i, j): stats(pick(g, "d%d_f%d" % (i, j), f), g["d%d_f%d" % (i, j)]) for i, fs in enumerate(res) for j, f in enumerate(fs)}


@functools.lru_cache(maxsize=None)
def tocgd_floor(name, precision):
    g = load_golden(name)
    seed = int(g["seed"])
    sd = synth_state_dict("tocgd", seed)
    i1, i2 = synth.tocg_inputs(1, 256, 192, seed)
    segs = synth.one_hot(synth.labels((1, 256, 192), 13, seed, "dseg"), 13)
    with torch.no_grad(), orc.storage_rounding(DT[precision]):
        res = orc.tocg_d_forward(sd, torch.cat([i1, i2, segs], 1))
    return {"d%d" % i: stats(r[0], g["d%d" % i]) for i, r in enumerate(res)}
