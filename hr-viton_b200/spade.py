"""Host side of the SPADE generator and its multiscale PatchGAN discriminator.

The classes keep the reference's public surface — constructor arguments, forward() signatures, attribute names and
state_dict keys (network_generator.py:9-49,75-316,318-433) — but their forward() is an orchestration of the C-ABI
kernels (hrviton_b200.ops): activations are pixel-major bf16, every torch.cat / nearest up-sampling / InstanceNorm /
modulation / LeakyReLU of the reference lives in a kernel prologue or epilogue.  torch supplies device memory,
streams and the parameter containers only.  CPU tensors are refused: there is no CPU path.
"""
import torch
import torch.nn as nn
from torch.nn import init
from torch.nn.utils import spectral_norm

from . import ops
from .ops import ACT_LRELU, ACT_NONE, ACT_RELU, ACT_TANH, Act


def _need_cuda(t, who):
    if not t.is_cuda:
        raise RuntimeError("%s: hrviton_b200 runs on sm_100a only — got a CPU tensor (there is no CPU fallback)" % who)


def _param_key(module):
    """Cache key of the derived (packed bf16 / folded BatchNorm) copies of a module's parameters and buffers.  `_version` catches
    eager in-place updates (optimizer.step, load_state_dict); ops.PARAM_GEN catches what `_version` cannot see — CUDA-graph replays
    of a captured optimiser step and `.data` edits — and is bumped by the trainers' replay()/step() and by `invalidate_caches()`."""
    return (ops.PARAM_GEN[0],) + tuple((p.data_ptr(), p._version) for p in list(module.parameters()) + list(module.buffers()))


def invalidate_caches():
    """Forget every packed-weight / folded-BatchNorm cache (call after editing parameters behind autograd's back)."""
    ops.PARAM_GEN[0] += 1


class BaseNetwork(nn.Module):
    """network_generator.py:9-49."""

    def print_network(self):
        n = sum(p.numel() for p in self.parameters())
        print("Network [{}] was created. Total number of parameters: {:.1f} million. "
              "To see the architecture, do print(network).".format(type(self).__name__, n / 1000000))

    def init_weights(self, init_type="normal", gain=0.02):
        fillers = {
            "normal": lambda w: init.normal_(w, 0.0, gain),
            "xavier": lambda w: init.xavier_normal_(w, gain=gain),
            "xavier_uniform": lambda w: init.xavier_uniform_(w, gain=1.0),
            "kaiming": lambda w: init.kaiming_normal_(w, a=0, mode="fan_in"),
            "orthogonal": lambda w: init.orthogonal_(w, gain=gain),
        }

        def visit(m):
            cls = type(m).__name__
            if "BatchNorm2d" in cls:
                if getattr(m, "weight", None) is not None:
                    init.normal_(m.weight.data, 1.0, gain)
                if getattr(m, "bias", None) is not None:
                    init.constant_(m.bias.data, 0.0)
            elif ("Conv" in cls or "Linear" in cls) and hasattr(m, "weight"):
                if init_type == "none":
                    m.reset_parameters()
                elif init_type in fillers:
                    fillers[init_type](m.weight.data)
                else:
                    raise NotImplementedError("initialization method '{}' is not implemented".format(init_type))
                if getattr(m, "bias", None) is not None:
                    init.constant_(m.bias.data, 0.0)

        self.apply(visit)

    def forward(self, *inputs):
        pass


class MaskNorm(nn.Module):
    """Present for API parity only (network_generator.py:52-72): never instantiated by the generator
    (every block is built with use_mask_norm=False) — no kernel exists for it."""

    def __init__(self, norm_nc):
        super().__init__()
        self.norm_layer = nn.InstanceNorm2d(norm_nc, affine=False)

    def forward(self, x, mask):
        raise NotImplementedError("MaskNorm is dead code in the reference generator and is out of scope (SURVEY.md §2 row 7)")


def _records_grad(module, x):
    """Whether a forward of `module` on `x` has to build an autograd graph."""
    return torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in module.parameters()))


def _sigma(conv, training):
    """Old-style torch spectral_norm (dim 0, 1 power iteration, eps 1e-12): in training mode u,v are refreshed in
    place without grad, sigma = u . (W v) with the gradient through W (network_generator.py:138-143; SURVEY.md §8 B5).
    u and v enter as copies: the next forward's refresh must not invalidate a graph still waiting for its backward."""
    wm = conv.weight_orig.reshape(conv.weight_orig.shape[0], -1)
    u, v = conv.weight_u, conv.weight_v
    if training:
        with torch.no_grad():
            v.copy_(torch.nn.functional.normalize(torch.mv(wm.t(), u), dim=0, eps=1e-12))
            u.copy_(torch.nn.functional.normalize(torch.mv(wm, v), dim=0, eps=1e-12))
    return torch.dot(u.detach().clone(), torch.mv(wm, v.detach().clone()))


def conv_weight(conv, training):
    """Effective fp32 weight of a conv container: W_orig / sigma when it is spectrally normalised, else its weight.
    Differentiable; inference callers detach it."""
    if hasattr(conv, "weight_orig"):
        return conv.weight_orig / _sigma(conv, training)
    return conv.weight


class SPADENorm(nn.Module):
    """Parameter container of one SPADE normalisation (network_generator.py:75-99).  Its arithmetic runs inside
    SPADEResBlock.forward: hrv_instnorm_stats + the SPADE epilogue of hrv_conv2d_fwd."""

    def __init__(self, opt, norm_type, norm_nc, label_nc):
        super().__init__()
        self.param_opt = opt
        self.noise_scale = nn.Parameter(torch.zeros(norm_nc))
        assert norm_type.startswith("alias")
        kind = norm_type[len("alias"):]
        if kind == "instance":
            self.param_free_norm = nn.InstanceNorm2d(norm_nc, affine=False)
        elif kind == "batch":
            self.param_free_norm = nn.BatchNorm2d(norm_nc, affine=False)
        elif kind == "mask":
            self.param_free_norm = MaskNorm(norm_nc)
        else:
            raise ValueError("'{}' is not a recognized parameter-free normalization type in SPADENorm".format(kind))
        self.kind = kind
        nhidden = 128
        self.conv_shared = nn.Sequential(nn.Conv2d(label_nc, nhidden, kernel_size=3, padding=1), nn.ReLU())
        self.conv_gamma = nn.Conv2d(nhidden, norm_nc, kernel_size=3, padding=1)
        self.conv_beta = nn.Conv2d(nhidden, norm_nc, kernel_size=3, padding=1)

    def forward(self, x, seg, misalign_mask=None):
        raise RuntimeError("SPADENorm is fused into SPADEResBlock.forward in hrviton_b200; call the block")

    def packed(self):
        """(gamma|beta interleaved PackedConv, interleaved bias, noise_scale); conv_shared is packed by the block, which
        merges the conv_shared of all its norms into one GEMM over the same segmentation map."""
        if self.kind != "instance":
            raise NotImplementedError("only 'aliasinstance' SPADE normalisation has a kernel (the reference's configuration)")
        gb = ops.pack_weight(self.conv_gamma.weight.detach(), (1, 1), interleave=self.conv_beta.weight.detach())
        gb_bias = torch.stack([self.conv_gamma.bias.detach(), self.conv_beta.bias.detach()], 1).reshape(-1).float().contiguous()
        return gb, gb_bias, self.noise_scale.detach().float().contiguous()


class SPADEResBlock(nn.Module):
    """network_generator.py:125-173."""

    def __init__(self, opt, input_nc, output_nc, use_mask_norm=True):
        super().__init__()
        self.param_opt = opt
        self.learned_shortcut = input_nc != output_nc
        middle_nc = min(input_nc, output_nc)
        self.conv_0 = nn.Conv2d(input_nc, middle_nc, kernel_size=3, padding=1)
        self.conv_1 = nn.Conv2d(middle_nc, output_nc, kernel_size=3, padding=1)
        if self.learned_shortcut:
            self.conv_s = nn.Conv2d(input_nc, output_nc, kernel_size=1, bias=False)
        subnorm_type = opt.norm_G
        if subnorm_type.startswith("spectral"):
            subnorm_type = subnorm_type[len("spectral"):]
            for name in ("conv_0", "conv_1") + (("conv_s",) if self.learned_shortcut else ()):
                setattr(self, name, spectral_norm(getattr(self, name)))
        label_nc = opt.gen_semantic_nc
        if use_mask_norm:
            subnorm_type, label_nc = "aliasmask", label_nc + 1
        self.norm_0 = SPADENorm(opt, subnorm_type, input_nc, label_nc)
        self.norm_1 = SPADENorm(opt, subnorm_type, middle_nc, label_nc)
        if self.learned_shortcut:
            self.norm_s = SPADENorm(opt, subnorm_type, input_nc, label_nc)
        self.relu = nn.LeakyReLU(0.2)
        self._cache_key = None
        self._cache = None

    def _packed(self):
        key = (_param_key(self), self.training)
        if self._cache_key != key or self.training:
            norms = ([self.norm_s] if self.learned_shortcut else []) + [self.norm_0, self.norm_1]
            # one conv_shared GEMM for all norms of the block: N = 128 * len(norms), same seg operand read once
            wsh = torch.cat([m.conv_shared[0].weight.detach() for m in norms], 0)
            if 9 * wsh.shape[1] <= 64:
                # few-channel label map: column (im2col) form, one K=64 block instead of nine K=16 taps; one 128-channel GEMM per
                # norm (<= 128 output channels keeps each on the pixel-N kernel) writing its slice of the shared actv buffer
                shared = [ops.pack_weight(ops.im2col_weight(m.conv_shared[0].weight.detach(), 64), (0, 0),
                                          flops_per_pixel=2.0 * m.conv_shared[0].weight.shape[0] * wsh.shape[1] * 9) for m in norms]
            else:
                shared = ops.pack_weight(wsh, (1, 1))
            c = {"shared": shared,
                 "shared_b": torch.cat([m.conv_shared[0].bias.detach() for m in norms], 0).float().contiguous(),
                 "n0": self.norm_0.packed(), "n1": self.norm_1.packed(),
                 "c0": ops.pack_weight(conv_weight(self.conv_0, self.training).detach(), (1, 1)),
                 "c1": ops.pack_weight(conv_weight(self.conv_1, self.training).detach(), (1, 1)),
                 "b0": self.conv_0.bias.detach().float().contiguous(), "b1": self.conv_1.bias.detach().float().contiguous()}
            if self.learned_shortcut:
                c["ns"] = self.norm_s.packed()
                c["cs"] = ops.pack_weight(conv_weight(self.conv_s, self.training).detach(), (0, 0))
            self._cache, self._cache_key = c, (_param_key(self), self.training)
        return self._cache

    @staticmethod
    def _spade(pk, actv, x0, x0_shift, x1, noise, act, stats=None):
        """act(InstanceNorm(x + noise*ns) * (1 + gamma(actv)) + beta(actv)) for the virtual tensor cat(up(x0), x1)."""
        gb, gb_b, ns = pk
        n, h, w = actv.n, actv.h, actv.w
        mean, rstd = stats if stats is not None else ops.instnorm_stats2(x0, x0_shift, x1, h, w, [noise], [ns])[0]
        c = x0.c + (x1.c if x1 is not None else 0)
        return ops.conv2d_spade(actv, gb, Act.empty(n, h, w, c), x0, x0_shift, x1, mean, rstd, noise, ns, gb_b, act)

    def run(self, x0, x0_shift, x1, seg, noise_fn, out_act=ACT_NONE):
        """x = cat(nearest_up2^x0_shift(x0), x1) is never materialised.  seg: Act at this block's resolution.
        noise_fn(n,h,w) -> fp32 (n,h,w) cuda; draw order norm_s, norm_0, norm_1 (network_generator.py:157-171)."""
        p = self._packed()
        n, h, w = seg.n, seg.h, seg.w
        if isinstance(p["shared"], list):
            cols = ops.im2col(seg, 3, 3, 1, k_pad=64)
            nsh = sum(pw.n_gemm for pw in p["shared"])
            actv = Act.empty(n, h, w, nsh)
            c0 = 0
            for pw in p["shared"]:
                ops.conv2d(cols, pw, actv.slice(c0, pw.n_gemm), act=ACT_RELU, shift=p["shared_b"][c0:c0 + pw.n_gemm])
                c0 += pw.n_gemm
        else:
            actv = ops.conv2d(seg, p["shared"], Act.empty(n, h, w, p["shared"].n_gemm), act=ACT_RELU, shift=p["shared_b"])
        k = 0
        if self.learned_shortcut:
            # norm_s and norm_0 normalise the same x with their own noise: one pass over the source tensors yields both statistics
            nz_s, nz_0 = noise_fn(n, h, w), noise_fn(n, h, w)
            st_s, st_0 = ops.instnorm_stats2(x0, x0_shift, x1, h, w, [nz_s, nz_0], [p["ns"][2], p["n0"][2]])
            hs = self._spade(p["ns"], actv.slice(0, 128), x0, x0_shift, x1, nz_s, ACT_NONE, stats=st_s)
            x_s = ops.conv2d(hs, p["cs"], Act.empty(n, h, w, p["cs"].n_gemm))
            k = 128
            h0 = self._spade(p["n0"], actv.slice(k, 128), x0, x0_shift, x1, nz_0, ACT_LRELU, stats=st_0)
        else:
            assert x0_shift == 0 and x1 is None
            x_s = x0
            h0 = self._spade(p["n0"], actv.slice(k, 128), x0, x0_shift, x1, noise_fn(n, h, w), ACT_LRELU)
        dx = ops.conv2d(h0, p["c0"], Act.empty(n, h, w, p["c0"].n_gemm), shift=p["b0"])
        h1 = self._spade(p["n1"], actv.slice(k + 128, 128), dx, 0, None, noise_fn(n, h, w), ACT_LRELU)
        return ops.conv2d(h1, p["c1"], Act.empty(n, h, w, p["c1"].n_gemm), shift=p["b1"], res=x_s, act=out_act)

    def forward(self, x, seg, misalign_mask=None):
        """Stand-alone use with NCHW fp32 tensors (the generator calls run() on pixel-major activations)."""
        _need_cuda(x, "SPADEResBlock")
        if misalign_mask is not None:
            raise NotImplementedError("misalign_mask / MaskNorm path is dead code in the reference (SURVEY.md §2 row 7)")
        with torch.no_grad():
            n, _, h, w = x.shape
            xa = ops.from_nchw(x.float())
            sa = ops.from_nchw(seg.float(), size=(h, w))
            noise_fn = getattr(self, "noise_source", None) or (lambda b, hh, ww: torch.randn(b, hh, ww, device=x.device))
            return self.run(xa, 0, None, sa, noise_fn).to_nchw()


class SPADEGenerator(BaseNetwork):
    """network_generator.py:176-245.  forward(x (N,input_nc,H,W), seg (N,gen_semantic_nc,H,W)) -> (N,3,H,W) in (-1,1)."""

    def __init__(self, opt, input_nc):
        super().__init__()
        self.num_upsampling_layers = opt.num_upsampling_layers
        self.param_opt = opt
        self.sh, self.sw = self.compute_latent_vector_size(opt)
        nf = opt.ngf
        self.conv_0 = nn.Conv2d(input_nc, nf * 16, kernel_size=3, padding=1)
        for i in range(1, 8):
            self.add_module("conv_{}".format(i), nn.Conv2d(input_nc, 16, kernel_size=3, padding=1))
        plan = [("head_0", nf * 16, nf * 16), ("G_middle_0", nf * 16 + 16, nf * 16), ("G_middle_1", nf * 16 + 16, nf * 16),
                ("up_0", nf * 16 + 16, nf * 8), ("up_1", nf * 8 + 16, nf * 4), ("up_2", nf * 4 + 16, nf * 2),
                ("up_3", nf * 2 + 16, nf)]
        if self.num_upsampling_layers == "most":
            plan.append(("up_4", nf + 16, nf // 2))
            nf = nf // 2
        for name, cin, cout in plan:
            self.add_module(name, SPADEResBlock(opt, cin, cout, use_mask_norm=False))
        self._blocks = [p[0] for p in plan]
        self.conv_img = nn.Conv2d(nf, 3, kernel_size=3, padding=1)
        self.up = nn.Upsample(scale_factor=2, mode="nearest")
        self.relu = nn.LeakyReLU(0.2)
        self.tanh = nn.Tanh()
        self.noise_source = None  # tests inject: callable(n, h, w) -> fp32 (n,h,w) cuda tensor
        self._pyr_key = None
        self._pyr = None

    def compute_latent_vector_size(self, opt):
        ups = {"normal": 5, "more": 6, "most": 7}
        if self.num_upsampling_layers not in ups:
            raise ValueError("opt.num_upsampling_layers '{}' is not recognized".format(self.num_upsampling_layers))
        k = ups[self.num_upsampling_layers]
        return opt.fine_height // 2 ** k, opt.fine_width // 2 ** k

    def _pyramid_packed(self):
        convs = [getattr(self, "conv_%d" % i) for i in range(8)] + [self.conv_img]
        key = (ops.PARAM_GEN[0],) + tuple((c.weight.data_ptr(), c.weight._version, c.bias._version) for c in convs)
        if key != self._pyr_key:
            self._pyr = [(ops.pack_weight(c.weight.detach(), (1, 1)), c.bias.detach().float().contiguous()) for c in convs]
            self._pyr_key = key
        return self._pyr

    def forward(self, x, seg):
        _need_cuda(x, "SPADEGenerator")
        if self.num_upsampling_layers != "most":
            raise NotImplementedError("only num_upsampling_layers='most' (the reference's configuration) is implemented")
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            try:
                from . import autograd_g
            except ImportError:
                raise NotImplementedError("SPADEGenerator backward is not implemented yet: call under torch.no_grad()")
            return autograd_g.generator_forward_train(self, x, seg)
        return self._forward_impl(x, seg)

    def _forward_impl(self, x, seg):
        with torch.no_grad():
            dev = x.device
            x = x.float()
            seg = seg.float()
            n = x.shape[0]
            noise_fn = self.noise_source or (lambda b, hh, ww: torch.randn(b, hh, ww, device=dev))
            pyr = self._pyramid_packed()
            sizes = [(self.sh * 2 ** i, self.sw * 2 ** i) for i in range(8)]
            feats, segs = [], []
            for i, (hh, ww) in enumerate(sizes):
                s = ops.from_nchw(x, c_pad=16, size=(hh, ww))
                pw, b = pyr[i]
                feats.append(ops.conv2d(s, pw, Act.empty(n, hh, ww, pw.n_gemm), shift=b))
                segs.append(ops.from_nchw(seg, size=(hh, ww)))
            # reference up-sampling schedule for 'most': one x2 before every block after head_0
            h = self.head_0.run(feats[0], 0, None, segs[0], noise_fn)
            for j, name in enumerate(self._blocks[1:]):
                last = j == len(self._blocks) - 2
                h = getattr(self, name).run(h, 1, feats[j + 1], segs[j + 1], noise_fn, out_act=ACT_LRELU if last else ACT_NONE)
            pw, b = pyr[8]
            out = torch.empty((n, 3, sizes[-1][0], sizes[-1][1]), dtype=torch.float32, device=dev)
            ops.conv2d(h, pw, out, act=ACT_TANH, shift=b, out_layout=ops.capi.NCHW)
            return out


# ------------------------------------------------------------------------------------------------ discriminator

def get_nonspade_norm_layer(norm_type="instance"):
    """network_generator.py:401-433: wraps a conv in spectral norm and/or appends a parameter-free norm layer."""

    def add_norm_layer(layer):
        sub = norm_type
        if norm_type.startswith("spectral"):
            layer = spectral_norm(layer)
            sub = norm_type[len("spectral"):]
        if sub == "none" or len(sub) == 0:
            return layer
        if getattr(layer, "bias", None) is not None:  # meaningless before a normalisation
            delattr(layer, "bias")
            layer.register_parameter("bias", None)
        cout = getattr(layer, "out_channels", None) or layer.weight.size(0)
        if sub == "batch":
            norm = nn.BatchNorm2d(cout, affine=True)
        elif sub == "instance":
            norm = nn.InstanceNorm2d(cout, affine=False)
        else:
            raise ValueError("normalization layer %s is not recognized" % sub)
        return nn.Sequential(layer, norm)

    return add_norm_layer


class NLayerDiscriminator(BaseNetwork):
    """network_generator.py:250-291: PatchGAN, 4x4 convs (stride 2 x n_layers_D, then stride 1 to 1 channel)."""

    def __init__(self, opt):
        super().__init__()
        self.no_ganFeat_loss = opt.no_ganFeat_loss
        nf = opt.ndf
        norm_layer = get_nonspade_norm_layer(opt.norm_D)
        if "batch" in opt.norm_D:
            raise NotImplementedError("norm_D with BatchNorm has no kernel; the reference uses 'spectralinstance'")
        input_nc = opt.gen_semantic_nc + 3
        groups = [[nn.Conv2d(input_nc, nf, kernel_size=4, stride=2, padding=2), nn.LeakyReLU(0.2, False)]]
        for _ in range(1, opt.n_layers_D):
            nf_prev, nf = nf, min(nf * 2, 512)
            groups.append([norm_layer(nn.Conv2d(nf_prev, nf, kernel_size=4, stride=2, padding=2)), nn.LeakyReLU(0.2, False)])
        groups.append([nn.Conv2d(nf, 1, kernel_size=4, stride=1, padding=2)])
        for i, g in enumerate(groups):
            self.add_module("model" + str(i), nn.Sequential(*g))

    def forward(self, input):
        _need_cuda(input, "NLayerDiscriminator")
        from . import autograd_g
        with torch.set_grad_enabled(_records_grad(self, input)):
            outs = autograd_g.patchgan_forward(list(self.children()), autograd_g.FromNCHW.apply(input.float(), None, None), self.training)
            res = [autograd_g.nchw(o) for o in outs]
        return res if not self.no_ganFeat_loss else res[-1]


class MultiscaleDiscriminator(BaseNetwork):
    """network_generator.py:293-316."""

    def __init__(self, opt):
        super().__init__()
        self.no_ganFeat_loss = opt.no_ganFeat_loss
        for i in range(opt.num_D):
            self.add_module("discriminator_%d" % i, NLayerDiscriminator(opt))

    def downsample(self, input):
        _need_cuda(input, "MultiscaleDiscriminator.downsample")
        return ops.avgpool3s2(ops.from_nchw(input.float())).to_nchw()

    def forward(self, input):
        _need_cuda(input, "MultiscaleDiscriminator")
        from . import autograd_g
        with torch.set_grad_enabled(_records_grad(self, input)):
            return autograd_g.discriminator_forward_train(self, input)


class GANLoss(nn.Module):
    """network_generator.py:318-398 (tiny elementwise reductions; plain torch — out of kernel scope, SURVEY §2 row 13)."""

    def __init__(self, gan_mode, target_real_label=1.0, target_fake_label=0.0, tensor=torch.FloatTensor):
        super().__init__()
        if gan_mode not in ("ls", "original", "w", "hinge"):
            raise ValueError("Unexpected gan_mode {}".format(gan_mode))
        self.real_label, self.fake_label = target_real_label, target_fake_label
        self.gan_mode = gan_mode
        self.Tensor = tensor

    def _target(self, like, is_real):
        return torch.full_like(like, self.real_label if is_real else self.fake_label)

    def loss(self, input, target_is_real, for_discriminator=True):
        if self.gan_mode == "original":
            return torch.nn.functional.binary_cross_entropy_with_logits(input, self._target(input, target_is_real))
        if self.gan_mode == "ls":
            return torch.nn.functional.mse_loss(input, self._target(input, target_is_real))
        if self.gan_mode == "hinge":
            if for_discriminator:
                margin = (input - 1) if target_is_real else (-input - 1)
                return -torch.mean(torch.clamp(margin, max=0.0))
            assert target_is_real, "The generator's hinge loss must be aiming for real"
            return -torch.mean(input)
        return -input.mean() if target_is_real else input.mean()

    def __call__(self, input, target_is_real, for_discriminator=True):
        if not isinstance(input, list):
            return self.loss(input, target_is_real, for_discriminator)
        total = 0
        for pred in input:
            if isinstance(pred, list):
                pred = pred[-1]
            l = self.loss(pred, target_is_real, for_discriminator)
            bs = 1 if l.dim() == 0 else l.size(0)
            total = total + torch.mean(l.view(bs, -1), dim=1)
        return total / len(input)
