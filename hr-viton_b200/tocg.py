"""Host side of the try-on condition generator ("tocg") and its stage-1 discriminator.

Public surface, attribute names and state_dict keys follow networks.py:13-198,302-453 of the reference; forward() is an
orchestration of the C-ABI kernels on pixel-major bf16 activations.  torch.cat is replaced by channel slices of shared
buffers, the bilinear 'up' 1x1 convolution is commuted below the up-sampling (both linear, weights of the lerp sum to 1),
eval-mode BatchNorm is folded into the conv epilogue, and the flow up-sample + normalise + base grid + grid_sample chain
is one kernel (hrv_flow_warp).
"""
import functools
import os

import numpy as np
import torch
import torch.nn as nn
from torch.nn.utils import spectral_norm

from . import ops
from .ops import ACT_RELU, Act
from .spade import _need_cuda, _param_key, _records_grad


def make_grid(N, iH, iW, opt=None):
    """networks.py:161-168 — kept for the callers (train_condition.py:241 uses a 3-argument form)."""
    gx = torch.linspace(-1.0, 1.0, iW).view(1, 1, iW, 1).expand(N, iH, -1, -1)
    gy = torch.linspace(-1.0, 1.0, iH).view(1, iH, 1, 1).expand(N, -1, iW, -1)
    grid = torch.cat([gx, gy], 3)
    return grid.cuda() if (opt is None or getattr(opt, "cuda", True)) and torch.cuda.is_available() else grid


class ResBlock(nn.Module):
    """networks.py:171-198: scale conv ('down' 3x3 s2 | 'same' 1x1 | 'up' bilinear x2 + 1x1), then
    relu(r + norm(conv3x3(relu(norm(conv3x3(r))))))."""

    def __init__(self, in_nc, out_nc, scale="down", norm_layer=nn.BatchNorm2d):
        super().__init__()
        use_bias = norm_layer == nn.InstanceNorm2d
        assert scale in ["up", "down", "same"], "ResBlock scale must be in 'up' 'down' 'same'"
        self.kind = scale
        if scale == "same":
            self.scale = nn.Conv2d(in_nc, out_nc, kernel_size=1, bias=True)
        elif scale == "up":
            self.scale = nn.Sequential(nn.Upsample(scale_factor=2, mode="bilinear"), nn.Conv2d(in_nc, out_nc, kernel_size=1, bias=True))
        else:
            self.scale = nn.Conv2d(in_nc, out_nc, kernel_size=3, stride=2, padding=1, bias=use_bias)
        self.block = nn.Sequential(
            nn.Conv2d(out_nc, out_nc, kernel_size=3, stride=1, padding=1, bias=use_bias), norm_layer(out_nc), nn.ReLU(inplace=True),
            nn.Conv2d(out_nc, out_nc, kernel_size=3, stride=1, padding=1, bias=use_bias), norm_layer(out_nc))
        self.relu = nn.ReLU(inplace=True)
        self.in_nc, self.out_nc = in_nc, out_nc
        self._cache_key = None
        self._cache = None

    @staticmethod
    def _fold_bn(bn, conv_bias):
        """Eval-mode BatchNorm as per-channel (scale, shift) of the conv epilogue (networks.py:189,192)."""
        if not isinstance(bn, nn.BatchNorm2d):
            raise NotImplementedError("ResBlock kernels cover norm_layer=nn.BatchNorm2d (the reference's configuration)")
        s = (bn.weight.detach() / torch.sqrt(bn.running_var + bn.eps)).float()
        t = (bn.bias.detach() - bn.running_mean * s).float()
        if conv_bias is not None:
            t = t + conv_bias.detach().float() * s
        return s.contiguous(), t.contiguous()

    def _packed(self, cin_total):
        key = (_param_key(self), cin_total)
        if key != self._cache_key:
            c = {}
            if self.kind == "down":
                w = self.scale.weight.detach()
                c["scale"] = ops.pack_s2d(w, 1)
                c["scale_b"] = self.scale.bias.detach().float().contiguous() if self.scale.bias is not None else None
            else:
                conv = self.scale if self.kind == "same" else self.scale[1]
                c["scale"] = ops.pack_weight(conv.weight.detach(), (0, 0), cin_total=cin_total)
                c["scale_b"] = conv.bias.detach().float().contiguous()
            c["w0"] = ops.pack_weight(self.block[0].weight.detach(), (1, 1))
            c["w1"] = ops.pack_weight(self.block[3].weight.detach(), (1, 1))
            c["bn0"] = self._fold_bn(self.block[1], self.block[0].bias)
            c["bn1"] = self._fold_bn(self.block[4], self.block[3].bias)
            self._cache, self._cache_key = c, key
        return self._cache

    def run(self, x, out=None, out_fp32_nchw=None):
        """x: Act (its view may span several concatenated producers). out: optional destination Act (a channel slice)."""
        p = self._packed(x.c)
        n = x.n
        if self.kind == "down":
            src = ops.space_to_depth(x)
            r = ops.conv2d(src, p["scale"], Act.empty(n, src.h, src.w, self.out_nc), shift=p["scale_b"])
        elif self.kind == "same":
            r = ops.conv2d(x, p["scale"], Act.empty(n, x.h, x.w, self.out_nc), shift=p["scale_b"])
        else:
            lo = ops.conv2d(x, p["scale"], Act.empty(n, x.h, x.w, self.out_nc), shift=p["scale_b"])
            r = ops.bilinear_up2_add(lo, None, Act.empty(n, 2 * x.h, 2 * x.w, self.out_nc))
        h = ops.conv2d(r, p["w0"], Act.empty(n, r.h, r.w, self.out_nc), act=ACT_RELU, scale=p["bn0"][0], shift=p["bn0"][1])
        if out_fp32_nchw is not None:
            return ops.conv2d(h, p["w1"], out_fp32_nchw, act=ACT_RELU, scale=p["bn1"][0], shift=p["bn1"][1], res=r,
                              out_layout=ops.capi.NCHW)
        if out is None:
            out = Act.empty(n, r.h, r.w, self.out_nc)
        return ops.conv2d(h, p["w1"], out, act=ACT_RELU, scale=p["bn1"][0], shift=p["bn1"][1], res=r)

    def forward(self, x):
        _need_cuda(x, "ResBlock")
        if self.training:
            # train-mode BatchNorm (batch statistics, running-stat update) lives in the autograd path (networks.py:188-198)
            from . import autograd_tocg
            from .autograd_g import FromNCHW
            y = autograd_tocg._resblock(self, FromNCHW.apply(x.float(), None, None))
            return y[..., :self.out_nc].permute(0, 3, 1, 2).float()
        with torch.no_grad():
            return self.run(ops.from_nchw(x.float())).to_nchw()


class ConditionGenerator(nn.Module):
    """networks.py:13-159.  forward(opt, input1, input2, upsample='bilinear') — also accepts the stale
    2-positional form tocg(input1, input2) used by train_generator.py:215 / train_condition.py:158."""

    def __init__(self, opt, input1_nc, input2_nc, output_nc, ngf=64, norm_layer=nn.BatchNorm2d):
        super().__init__()
        self.warp_feature = opt.warp_feature
        self.out_layer_opt = opt.out_layer
        self._opt = opt
        rb = functools.partial(ResBlock, norm_layer=norm_layer)
        enc = [ngf, ngf * 2, ngf * 4, ngf * 4, ngf * 4]
        self.ClothEncoder = nn.Sequential(*[rb(i, o, scale="down") for i, o in zip([input1_nc] + enc[:-1], enc)])
        self.PoseEncoder = nn.Sequential(*[rb(i, o, scale="down") for i, o in zip([input2_nc] + enc[:-1], enc)])
        self.conv = rb(ngf * 4, ngf * 8, scale="same")
        if opt.warp_feature == "T1":
            dec_in = [ngf * 8, ngf * 4 * 2 + ngf * 4, ngf * 4 * 2 + ngf * 4, ngf * 2 * 2 + ngf * 4, ngf * 1 * 2 + ngf * 4]
        elif opt.warp_feature == "encoder":
            dec_in = [ngf * 8, ngf * 4 * 3, ngf * 4 * 3, ngf * 2 * 3, ngf * 1 * 3]
        else:
            raise ValueError("unknown warp_feature %r" % (opt.warp_feature,))
        dec_out = [ngf * 4, ngf * 4, ngf * 2, ngf, ngf]
        self.SegDecoder = nn.Sequential(*[rb(i, o, scale="up") for i, o in zip(dec_in, dec_out)])
        if opt.out_layer == "relu":
            self.out_layer = rb(ngf + input1_nc + input2_nc, output_nc, scale="same")
        elif opt.out_layer == "conv":
            self.out_layer = nn.Sequential(rb(ngf + input1_nc + input2_nc, ngf, scale="same"), nn.Conv2d(ngf, output_nc, kernel_size=1, bias=True))
        lat = [ngf, ngf * 2, ngf * 4, ngf * 4]
        self.conv1 = nn.Sequential(*[nn.Conv2d(c, ngf * 4, kernel_size=1, bias=True) for c in lat])
        self.conv2 = nn.Sequential(*[nn.Conv2d(c, ngf * 4, kernel_size=1, bias=True) for c in lat])  # dead in forward (networks.py:131)
        self.flow_conv = nn.ModuleList([nn.Conv2d(ngf * 8, 2, kernel_size=3, stride=1, padding=1, bias=True) for _ in range(5)])
        self.bottleneck = nn.Sequential(*[nn.Sequential(nn.Conv2d(c, ngf * 4, kernel_size=3, stride=1, padding=1, bias=True), nn.ReLU())
                                          for c in [ngf * 4, ngf * 4, ngf * 2, ngf]])
        self.ngf = ngf
        self.io = (input1_nc, input2_nc, output_nc)
        self._cache_key = None
        self._cache = None

    def normalize(self, x):
        return x

    def _packed(self):
        mods = [self.conv1, self.flow_conv, self.bottleneck]
        key = tuple(_param_key(m) for m in mods)
        if key != self._cache_key:
            c = {"conv1": [(ops.pack_weight(m.weight.detach(), (0, 0)), m.bias.detach().float().contiguous()) for m in self.conv1],
                 "flow": [(ops.pack_weight(m.weight.detach(), (1, 1)), m.bias.detach().float().contiguous()) for m in self.flow_conv],
                 "bott": [(ops.pack_weight(m[0].weight.detach(), (1, 1)), m[0].bias.detach().float().contiguous()) for m in self.bottleneck]}
            self._cache, self._cache_key = c, key
        return self._cache

    def forward(self, *args, **kwargs):
        args = list(args)
        if args and not torch.is_tensor(args[0]):
            args.pop(0)  # the `opt` positional of the reference signature; the ctor-time opt carries the same fields
        input1, input2 = args[0], args[1]
        upsample = args[2] if len(args) > 2 else kwargs.get("upsample", "bilinear")
        if upsample != "bilinear":
            raise NotImplementedError("only upsample='bilinear' (the reference default, the only value any caller passes)")
        _need_cuda(input1, "ConditionGenerator")
        if self.warp_feature != "T1" or self.out_layer_opt != "relu":
            raise NotImplementedError("kernels cover warp_feature='T1', out_layer='relu' (the reference's configuration)")
        if self.training:
            # train mode = batch-statistics BatchNorm (+ running-stat updates) exactly as nn.BatchNorm2d in the reference
            # (train_condition.py:158 calls tocg(input1, input2) in train mode); with grad enabled it also carries the autograd graph
            from . import autograd_tocg
            return autograd_tocg.tocg_forward_train(self, input1, input2)
        if torch.is_grad_enabled() and (input1.requires_grad or input2.requires_grad):
            raise NotImplementedError("eval-mode ConditionGenerator is inference only (folded BatchNorm): no gradient w.r.t. its inputs; "
                                      "call .train() for the differentiable path or wrap the call in torch.no_grad()")
        with torch.no_grad():
            return self._forward_impl(input1.float().contiguous(), input2.float().contiguous())

    def _forward_impl(self, input1, input2):
        P = self._packed()
        n, c1, H, W = input1.shape
        c2 = input2.shape[1]
        ngf = self.ngf
        dev = input1.device
        # --- decoder concat buffers, one per pyramid level lvl (resolution of E*[lvl]):  [x | E2[lvl] | warped_T1 | bott]
        enc_c = [ngf, ngf * 2, ngf * 4, ngf * 4, ngf * 4]
        dec_out = [ngf * 4, ngf * 4, ngf * 2, ngf, ngf]  # x channels arriving at lvl = 3,2,1,0 are dec_out[0..3]
        res = [(H >> (k + 1), W >> (k + 1)) for k in range(5)]
        cat = {}
        for i in range(1, 5):
            lvl = 4 - i
            cx = dec_out[i - 1]
            cat[lvl] = (Act.empty(n, res[lvl][0], res[lvl][1], cx + enc_c[lvl] + 2 * ngf * 4), cx)
        a1 = ops.from_nchw(input1)
        # final concat [x(ngf) | input2 | warped_input1]
        fin = Act.empty(n, H, W, ngf + c2 + c1, zero=True)
        ops.from_nchw(input2, out=fin.slice(ngf, c2))
        a2 = fin.slice(ngf, c2)
        # --- encoders (networks.py:105-111)
        e1, e2 = [], []
        bott0 = Act.empty(n, res[4][0], res[4][1], 2 * ngf * 4)  # [T1 | T2] at the coarsest level (E4, networks.py:121)
        xa, xb = a1, a2
        for k in range(5):
            if k == 4:
                o1, o2 = bott0.slice(0, ngf * 4), bott0.slice(ngf * 4, ngf * 4)
            else:
                o1 = None
                buf, cx = cat[k]
                o2 = buf.slice(cx, enc_c[k])
            xa = self.ClothEncoder[k].run(xa, out=o1)
            xb = self.PoseEncoder[k].run(xb, out=o2)
            e1.append(xa)
            e2.append(xb)
        # --- coarsest level
        flows = []
        pw, b = P["flow"][0]
        f0 = Act.empty(n, res[4][0], res[4][1], 2, dtype=torch.float32, pitch=2)
        ops.conv2d(bott0, pw, f0, shift=b)
        flows.append(f0.buf)
        x = self.conv.run(e2[4])
        buf, cx = cat[3]
        x = self.SegDecoder[0].run(x, out=buf.slice(0, cx))
        t1 = e1[4]
        # --- refinement levels (networks.py:129-145)
        for i in range(1, 5):
            lvl = 4 - i
            hh, ww = res[lvl]
            buf, cx = cat[lvl]
            ce = enc_c[lvl]
            pw, b = P["conv1"][lvl]
            lat = ops.conv2d(e1[lvl], pw, Act.empty(n, hh, ww, ngf * 4), shift=b)
            t1 = ops.bilinear_up2_add(t1, lat, Act.empty(n, hh, ww, ngf * 4))
            warped = buf.slice(cx + ce, ngf * 4)
            flow_up, _ = ops.flow_warp(flows[-1], t1, warped)
            pw, b = P["bott"][i - 1]
            ops.conv2d(buf.slice(0, cx), pw, buf.slice(cx + ce + ngf * 4, ngf * 4), act=ACT_RELU, shift=b)
            pw, b = P["flow"][i]
            f = Act.empty(n, hh, ww, 2, dtype=torch.float32, pitch=2)
            ops.conv2d(buf.slice(cx + ce, 2 * ngf * 4), pw, f, shift=b, res=Act(flow_up))
            flows.append(f.buf)
            dec_in = buf.slice(0, cx + ce + ngf * 4)
            if i < 4:
                nbuf, ncx = cat[lvl - 1]
                x = self.SegDecoder[i].run(dec_in, out=nbuf.slice(0, ncx))
            else:
                x = self.SegDecoder[i].run(dec_in, out=fin.slice(0, ngf))
        # --- full resolution: warp input1 (cloth + mask) with the last flow (networks.py:147-152)
        src32 = Act(input1.permute(0, 2, 3, 1).contiguous())
        w32 = Act.empty(n, H, W, c1, dtype=torch.float32, pitch=c1)
        ops.flow_warp(flows[-1], src32, w32, want_flow_up=False)
        ops.flow_warp(flows[-1], a1, fin.slice(ngf + c2, c1), want_flow_up=False)
        seg = torch.empty((n, self.io[2], H, W), dtype=torch.float32, device=dev)
        self.out_layer.run(fin, out_fp32_nchw=seg)
        warped_in = w32.buf.permute(0, 3, 1, 2)
        return flows, seg, warped_in[:, :-1].contiguous(), warped_in[:, -1:].contiguous()


# ------------------------------------------------------------------------------------------------ stage-1 discriminator

class NLayerDiscriminator(nn.Module):
    """networks.py:351-408."""

    def __init__(self, input_nc, ndf=64, n_layers=3, norm_layer=nn.BatchNorm2d, use_sigmoid=False, getIntermFeat=False,
                 Ddropout=False, spectral=False):
        super().__init__()
        self.getIntermFeat = getIntermFeat
        self.n_layers = n_layers
        sn = spectral_norm if spectral else (lambda m: m)
        self.spectral_norm = sn
        kw, padw = 4, int(np.ceil((4 - 1.0) / 2))
        groups = [[nn.Conv2d(input_nc, ndf, kernel_size=kw, stride=2, padding=padw), nn.LeakyReLU(0.2, True)]]
        nf = ndf
        for _ in range(1, n_layers):
            nf_prev, nf = nf, min(nf * 2, 512)
            g = [sn(nn.Conv2d(nf_prev, nf, kernel_size=kw, stride=2, padding=padw)), norm_layer(nf), nn.LeakyReLU(0.2, True)]
            if Ddropout:
                g.append(nn.Dropout(0.5))
            groups.append(g)
        nf_prev, nf = nf, min(nf * 2, 512)
        groups.append([nn.Conv2d(nf_prev, nf, kernel_size=kw, stride=1, padding=padw), norm_layer(nf), nn.LeakyReLU(0.2, True)])
        groups.append([nn.Conv2d(nf, 1, kernel_size=kw, stride=1, padding=padw)])
        if use_sigmoid:
            groups.append([nn.Sigmoid()])
        if getIntermFeat:
            for i, g in enumerate(groups):
                setattr(self, "model" + str(i), nn.Sequential(*g))
        else:
            self.model = nn.Sequential(*[m for g in groups for m in g])

    def forward(self, input):
        _need_cuda(input, "NLayerDiscriminator")
        from . import autograd_g
        seqs = [getattr(self, "model" + str(i)) for i in range(self.n_layers + 2)] if self.getIntermFeat else [self.model]
        with torch.set_grad_enabled(_records_grad(self, input)):
            outs = autograd_g.patchgan_forward(seqs, autograd_g.FromNCHW.apply(input.float(), None, None), self.training)
            res = [autograd_g.nchw(o) for o in outs]
        return res if self.getIntermFeat else res[-1]


class MultiscaleDiscriminator(nn.Module):
    """networks.py:302-349."""

    def __init__(self, input_nc, ndf=64, n_layers=3, norm_layer=nn.BatchNorm2d, use_sigmoid=False, num_D=3, getIntermFeat=False,
                 Ddownx2=False, Ddropout=False, spectral=False):
        super().__init__()
        self.num_D, self.n_layers, self.getIntermFeat, self.Ddownx2 = num_D, n_layers, getIntermFeat, Ddownx2
        for i in range(num_D):
            netD = NLayerDiscriminator(input_nc, ndf, n_layers, norm_layer, use_sigmoid, getIntermFeat, Ddropout, spectral=spectral)
            if getIntermFeat:
                for j in range(n_layers + 2):
                    setattr(self, "scale" + str(i) + "_layer" + str(j), getattr(netD, "model" + str(j)))
            else:
                setattr(self, "layer" + str(i), netD.model)
        self.downsample = nn.AvgPool2d(3, stride=2, padding=[1, 1], count_include_pad=False)

    def forward(self, input):
        _need_cuda(input, "MultiscaleDiscriminator")
        # train_condition.py:208-232: D(fake) back-propagates into tocg, D(real / fake.detach()) into D
        from . import autograd_tocg
        with torch.set_grad_enabled(_records_grad(self, input)):
            return autograd_tocg.tocg_discriminator_forward_train(self, input)


def weights_init(m):
    """networks.py:428-435."""
    name = type(m).__name__
    if name.find("Conv2d") != -1:
        m.weight.data.normal_(0.0, 0.02)
    elif name.find("BatchNorm2d") != -1:
        m.weight.data.normal_(1.0, 0.02)
        m.bias.data.fill_(0)


def get_norm_layer(norm_type="instance"):
    if norm_type == "batch":
        return functools.partial(nn.BatchNorm2d, affine=True)
    if norm_type == "instance":
        return functools.partial(nn.InstanceNorm2d, affine=False)
    raise NotImplementedError("normalization layer [%s] is not found" % norm_type)


def define_D(input_nc, ndf=64, n_layers_D=3, norm="instance", use_sigmoid=False, num_D=2, getIntermFeat=False, gpu_ids=[],
             Ddownx2=False, Ddropout=False, spectral=False):
    """networks.py:445-453."""
    netD = MultiscaleDiscriminator(input_nc, ndf, n_layers_D, get_norm_layer(norm), use_sigmoid, num_D, getIntermFeat,
                                   Ddownx2, Ddropout, spectral=spectral)
    print(netD)
    if len(gpu_ids) > 0:
        assert torch.cuda.is_available()
        netD.cuda()
    netD.apply(weights_init)
    return netD


def save_checkpoint(model, save_path, opt=None):
    """networks.py:411-417."""
    d = os.path.dirname(save_path)
    if d and not os.path.exists(d):
        os.makedirs(d)
    torch.save(model.cpu().state_dict(), save_path)
    if opt is None or getattr(opt, "cuda", True):
        model.cuda()


def load_checkpoint(model, checkpoint_path, opt=None):
    """networks.py:419-425 (missing file -> raises, as the reference's bare `raise` does)."""
    if not os.path.exists(checkpoint_path):
        print("no checkpoint")
        raise FileNotFoundError(checkpoint_path)
    model.load_state_dict(torch.load(checkpoint_path), strict=False)
    if opt is None or getattr(opt, "cuda", True):
        model.cuda()
