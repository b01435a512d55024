"""Generates tests/golden/*.npz by running the UNMODIFIED reference modules
(imported from a checkout of sangyun884/HR-VITON, CPU fp32) on deterministic synthetic
weights and inputs (hrviton_b200.synth):

    python tests/golden/make_golden.py --reference <HR-VITON checkout>

The tests need no checkout: they re-create the same weights/inputs from the seeds
stored in each fixture and compare against the stored outputs.  Every fixture stays
under 1 MB: an output with more than `cap` elements per image is stored as a fixed
per-image sample (sample_large), its flat per-image indices next to it as `<key>_idx`.
"""
import argparse
import os
import sys
import types
import zlib

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
import hrv_loader  # noqa: E402

hrv_loader.load()
from hrviton_b200 import synth  # noqa: E402


def import_reference(ref):
    ref = os.path.abspath(ref)
    sys.path.insert(0, ref)
    import importlib
    ref_networks = importlib.import_module("networks")
    ref_gen = importlib.import_module("network_generator")
    sys.path.remove(ref)
    assert ref_networks.__file__.startswith(ref) and ref_gen.__file__.startswith(ref)
    return ref_networks, ref_gen


def tocg_opt():
    return types.SimpleNamespace(warp_feature="T1", out_layer="relu", cuda=False)


def gen_opt(h, w):
    return types.SimpleNamespace(norm_G="spectralaliasinstance", gen_semantic_nc=7, ngf=64,
                                 num_upsampling_layers="most", fine_height=h, fine_width=w, cuda=False,
                                 ndf=64, norm_D="spectralinstance", n_layers_D=3, num_D=2, no_ganFeat_loss=False)


# elements per image kept of each output (sample_large), per fixture: what keeps the file under 1 MB
CAPS = {"tocg_256x192_b1": 90112, "tocg_128x96_b2": 98304, "gen_512x384_b1": 262144, "gend_128x96_b2": 16384,
        "gen_1024x768_b8": 28672, "tocg_1024x768_b4": 9216}


def sample_large(arrs, cap):
    """Floating-point outputs with more than `cap` elements per image (leading dim = batch) become (N, cap): the same `cap` positions
    of every image, drawn once per key from a generator seeded by the key's name; their sorted flat indices are stored as `<key>_idx`
    (tests/helpers.pick applies them to the computed output)."""
    out = {}
    for k, v in arrs.items():
        a = v.detach().numpy() if torch.is_tensor(v) else np.asarray(v)
        if cap is not None and a.dtype.kind == "f" and a.ndim > 1 and a[0].size > cap:
            idx = np.sort(np.random.default_rng(zlib.crc32(k.encode())).choice(a[0].size, cap, replace=False)).astype(np.int32)
            out[k + "_idx"] = idx
            a = a.reshape(a.shape[0], -1)[:, idx]
        out[k] = a
    return out


def save(name, **arrs):
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **sample_large(arrs, CAPS.get(name)))
    print("wrote", path, "%.2f MB" % (os.path.getsize(path) / 1e6))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", required=True, help="checkout of the original HR-VITON repository")
    ap.add_argument("--only", default="")
    args = ap.parse_args()
    torch.set_num_threads(os.cpu_count())
    ref_networks, ref_gen = import_reference(args.reference)
    torch.manual_seed(0)

    def want(n):
        return (not args.only and n != "big") or args.only == n

    with torch.no_grad():
        if want("tocg"):
            for tag, (n, h, w) in {"tocg_256x192_b1": (1, 256, 192), "tocg_128x96_b2": (2, 128, 96)}.items():
                seed = 11
                m = ref_networks.ConditionGenerator(tocg_opt(), 4, 16, 13, ngf=96, norm_layer=torch.nn.BatchNorm2d).eval()
                sd = m.state_dict()
                synth.fill_state_dict(sd, seed)
                m.load_state_dict(sd)
                i1, i2 = synth.tocg_inputs(n, h, w, seed)
                flows, seg, wc, wcm = m(tocg_opt(), i1, i2)
                save(tag, seed=seed, shape=[n, h, w], seg=seg, warped_c=wc, warped_cm=wcm,
                     **{"flow%d" % i: f for i, f in enumerate(flows)})

        if want("gen"):
            for tag, (n, h, w) in {"gen_512x384_b1": (1, 512, 384), "gen_256x256_b2": (2, 256, 256)}.items():
                seed = 23
                opt = gen_opt(h, w)
                m = ref_gen.SPADEGenerator(opt, 9).eval()
                sd = m.state_dict()
                synth.fill_state_dict(sd, seed)
                m.load_state_dict(sd)
                x, seg = synth.gen_inputs(n, h, w, seed)
                counter = [0]
                real_randn = torch.randn

                def fake_randn(b, ww, hh, one, *a, **k):
                    t = synth.spade_noise(b, hh, ww, seed, counter[0])  # (N,H,W)
                    counter[0] += 1
                    return t[:, None].transpose(1, 3).contiguous()  # back to (b,w,h,1)

                torch.randn = fake_randn
                try:
                    out = m(x, seg)
                finally:
                    torch.randn = real_randn
                save(tag, seed=seed, shape=[n, h, w], out=out.half(), n_noise=counter[0])  # fp16 storage: 5e-4 abs on (-1,1)

        if want("big"):
            # ---- the BENCHMARKED shapes (BASELINE.json configs 2-4): 1024x768, generator batch 8, tocg batch 4.  Full outputs
            # would be 75 MB; the fixture keeps a stride-8 sub-sampling of every output, four full-resolution 64x64 crops and
            # per-image per-channel sums (fp64) — enough to catch tile-addressing errors anywhere in the >2^31-byte buffers.
            seed = 23
            n, h, w = 8, 1024, 768
            m = ref_gen.SPADEGenerator(gen_opt(h, w), 9).eval()
            sd = m.state_dict()
            synth.fill_state_dict(sd, seed)
            m.load_state_dict(sd)
            x, seg = synth.gen_inputs(n, h, w, seed)
            outs = []
            real_randn = torch.randn
            for i in range(n):  # eval mode is per-sample independent: one image at a time keeps the CPU footprint small
                counter = [0]

                def fake_randn(b, ww, hh, one, *a, **k):
                    t = synth.spade_noise(n, hh, ww, seed, counter[0])[i:i + 1]  # image i's slice of the batch-8 draw
                    counter[0] += 1
                    return t[:, None].transpose(1, 3).contiguous()

                torch.randn = fake_randn
                try:
                    outs.append(m(x[i:i + 1], seg[i:i + 1]))
                finally:
                    torch.randn = real_randn
                print("gen big image", i, flush=True)
            out = torch.cat(outs, 0)
            crops = [(0, 0), (0, w - 64), (h - 64, 0), (h // 2 - 32, w // 2 - 32)]
            save("gen_1024x768_b8", seed=seed, shape=[n, h, w], sub8=out[:, :, ::8, ::8].half(),
                 crops=torch.stack([out[:, :, y:y + 64, x0:x0 + 64] for y, x0 in crops], 1).half(), crop_yx=np.asarray(crops),
                 chan_sums=out.double().sum((2, 3)))
            seed = 11
            n = 4
            m = ref_networks.ConditionGenerator(tocg_opt(), 4, 16, 13, ngf=96, norm_layer=torch.nn.BatchNorm2d).eval()
            sd = m.state_dict()
            synth.fill_state_dict(sd, seed)
            m.load_state_dict(sd)
            i1, i2 = synth.tocg_inputs(n, h, w, seed)
            flows, sg, wc, wcm = m(tocg_opt(), i1, i2)
            save("tocg_1024x768_b4", seed=seed, shape=[n, h, w], seg_sub8=sg[:, :, ::8, ::8], seg_sums=sg.double().sum((2, 3)),
                 seg_crop=sg[:, :, h - 64:, w - 64:], warped_c_sub8=wc[:, :, ::8, ::8], warped_cm_sub8=wcm[:, :, ::8, ::8],
                 **{"flow%d_sub" % i: f[:, ::(1 if i < 3 else 4), ::(1 if i < 3 else 4)] for i, f in enumerate(flows)})

        if want("gend"):
            seed = 31
            opt = gen_opt(256, 192)
            m = ref_gen.MultiscaleDiscriminator(opt).eval()
            sd = m.state_dict()
            synth.fill_state_dict(sd, seed)
            m.load_state_dict(sd)
            x, seg = synth.gen_inputs(2, 128, 96, seed, input_nc=3)
            res = m(torch.cat([seg, x], 1))
            save("gend_128x96_b2", seed=seed, shape=[2, 128, 96],
                 **{"d%d_f%d" % (i, j): f for i, fs in enumerate(res) for j, f in enumerate(fs)})

        if want("tocgd"):
            seed = 37
            m = ref_networks.define_D(input_nc=33, Ddownx2=True, Ddropout=True, n_layers_D=3, spectral=False, num_D=2).eval()
            sd = m.state_dict()
            synth.fill_state_dict(sd, seed)
            m.load_state_dict(sd)
            i1, i2 = synth.tocg_inputs(1, 256, 192, seed)
            segs = synth.one_hot(synth.labels((1, 256, 192), 13, seed, "dseg"), 13)
            res = m(torch.cat([i1, i2, segs], 1))
            save("tocgd_256x192_b1", seed=seed, shape=[1, 256, 192], **{"d%d" % i: r[0] for i, r in enumerate(res)})


if __name__ == "__main__":
    main()
