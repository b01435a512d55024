"""Training path (forward + backward) of the SPADE generator, and the one forward of both PatchGAN discriminators.

torch.autograd carries the graph; every node is a fused C-ABI op on pixel-major bf16 buffers:

  ConvFn    y = act(conv(x, W) * 1 + b (+ res))          fwd: hrv_conv2d_fwd
            dX  = conv(dY', flip(W)^T)                     bwd: hrv_conv2d_fwd again (dgrad IS a convolution)
            dW  = x^T (*) dY'                              bwd: hrv_conv2d_wgrad (tcgen05, pixel-K GEMM with MN-major operands)
  SpadeFn   h = act(IN(cat(up(x0),x1) + noise*ns) * (1+gamma(actv)) + beta(actv))
            fwd: hrv_instnorm_stats + hrv_conv2d_fwd(SPADE epilogue); bwd: modulation / InstanceNorm backward +
            dgrad/wgrad of the gamma|beta GEMM.

Spectral norm stays differentiable in torch (W/sigma with sigma = u.(W v), tiny weight-sized tensors), exactly as the
reference's old-style torch.nn.utils.spectral_norm does (network_generator.py:138-143).
"""
import os

import torch
import torch.nn.functional as F

from . import ops
from .ops import ACT_LRELU, ACT_NONE, ACT_RELU, ACT_TANH, Act, im2col_weight
from .spade import conv_weight


def _act_grad(dy, y, act):
    """dL/dv from dL/dy for y = act(v), using only y (all our activations are invertible in sign / value)."""
    if act == ACT_NONE:
        return dy
    if act == ACT_RELU:
        return dy * (y > 0).to(dy.dtype)
    if act == ACT_LRELU:
        return torch.where(y > 0, dy, dy * 0.2)
    if act == ACT_TANH:
        return dy * (1 - y.float() * y.float()).to(dy.dtype)
    raise ValueError(act)


def _wgrad(x_buf, cin, dy_buf, cout, kh, kw, pad):
    """dW (cout,cin,kh,kw) fp32 = sum over pixels of dY[p,co] * X[p+tap-pad,ci] on tcgen05 (hrv_conv2d_wgrad).
    HRV_WGRAD=cudnn selects the library weight-gradient instead (A/B comparisons only)."""
    if os.environ.get("HRV_WGRAD") == "cudnn":
        x = x_buf[..., :cin].permute(0, 3, 1, 2)
        dy = dy_buf[..., :cout].permute(0, 3, 1, 2)
        return torch.nn.grad.conv2d_weight(x, (cout, cin, kh, kw), dy, stride=1, padding=pad).float()
    return ops.conv2d_wgrad(Act(x_buf, c=cin), Act(dy_buf, c=cout), kh, kw, pad)


class ConvFn(torch.autograd.Function):
    """y = act(conv(x_buf[..., :cin], w, padding=pad) + bias (+ res_buf)) on (N,H,W,P) bf16 buffers, stride 1.
    Output extent = H + 2*pad - kh + 1 ('same' for 3x3/1, 1x1/0; H+1 for the PatchGAN 4x4/2 and 2x2/1 forms).
    need_wgrad=False skips dW (frozen nets: VGG, D inside the G step)."""

    @staticmethod
    def forward(ctx, x_buf, w, bias, res_buf, act, out_fp32_nchw, pad, out_f32_nhwc, out_hw=None, gate_in=ACT_NONE, gated_out=False):
        """gate_in: x_buf is the saved OUTPUT of a layer with that activation whose backward this node's data-gradient convolution
        applies in its epilogue (dx *= act'(x_buf)).  gated_out: every consumer of y applies this node's activation backward itself, so
        backward() receives dL/dv directly.  Together they remove the dv = dy * act'(y) pass from ReLU chains (Vgg19)."""
        cout, cin, kh, kw = w.shape
        n, h, wd, _ = x_buf.shape
        oh, ow = h + 2 * pad - kh + 1, wd + 2 * pad - kw + 1
        if out_hw is not None:  # cropped output (top-left aligned): rows/columns beyond it are never computed
            assert out_hw[0] <= oh and out_hw[1] <= ow
            oh, ow = out_hw
        xa = Act(x_buf, c=cin)
        pw = ops.pack_weight(w.detach(), (pad, pad))
        b = bias.detach().float().contiguous() if bias is not None else None
        res = Act(res_buf, c=cout) if res_buf is not None else None
        if out_fp32_nchw:
            y = torch.empty((n, cout, oh, ow), dtype=torch.float32, device=x_buf.device)
            ops.conv2d(xa, pw, y, act=act, shift=b, res=res, out_layout=ops.capi.NCHW)
        elif out_f32_nhwc:
            ya = Act.empty(n, oh, ow, cout, dtype=torch.float32, pitch=cout)
            ops.conv2d(xa, pw, ya, act=act, shift=b, res=res)
            y = ya.buf
        else:
            ya = Act.empty(n, oh, ow, cout)
            ops.conv2d(xa, pw, ya, act=act, shift=b, res=res)
            y = ya.buf
        ctx.save_for_backward(x_buf, w, y if (act != ACT_NONE and not gated_out) else None)
        ctx.meta = (act if not gated_out else ACT_NONE, out_fp32_nchw, bias is not None, res_buf is not None, pad, out_f32_nhwc)
        ctx.gate_in = gate_in
        return y

    @staticmethod
    def backward(ctx, dy):
        x_buf, w, y = ctx.saved_tensors
        act, nchw, has_bias, has_res, pad, f32_nhwc = ctx.meta
        cout, cin, kh, kw = w.shape
        db = None
        if nchw:  # fp32 NCHW upstream gradient (image output): bring it to the pixel-major bf16 convention
            dv32 = _act_grad(dy, y, act).float()
            if has_bias and ctx.needs_input_grad[2]:
                db = dv32.sum((0, 2, 3))
            dv_buf = ops.from_nchw(dv32.contiguous()).buf
        elif f32_nhwc:
            dv = _act_grad(dy, y, act)
            if has_bias and ctx.needs_input_grad[2]:
                db = dv.sum((0, 1, 2), dtype=torch.float32)
            dv_buf = torch.zeros(dv.shape[:3] + (ops.round_up(cout, 8),), dtype=x_buf.dtype, device=dv.device)
            dv_buf[..., :cout] = dv.to(x_buf.dtype)
        else:  # one fused pass: activation backward + bias gradient
            want_b = has_bias and ctx.needs_input_grad[2]
            dva, db = ops.act_bwd_bias(Act(dy.contiguous(), c=cout), Act(y, c=cout) if y is not None else None, act, want_bias=want_b)
            dv_buf = dva.buf
        n, h, wd, _ = x_buf.shape
        dx = dw = dres = None
        if ctx.needs_input_grad[0]:
            pw = ops.pack_weight(w, (kh - 1 - pad, kw - 1 - pad), dgrad=True)  # flipped/transposed operand, packed in one kernel
            dxa = Act.empty(n, h, wd, cin, pitch=x_buf.shape[3], zero=x_buf.shape[3] > ops.round_up(cin, 8))
            if ctx.gate_in != ACT_NONE:  # activation backward of the producer of x_buf, fused into this convolution's epilogue
                mode = {ACT_RELU: ops.capi.RES_GATE_RELU, ACT_LRELU: ops.capi.RES_GATE_LRELU}[ctx.gate_in]
                ops.conv2d(Act(dv_buf, c=cout), pw, dxa, res=Act(x_buf, c=cin), res_mode=mode)
            else:
                ops.conv2d(Act(dv_buf, c=cout), pw, dxa)
            dx = dxa.buf
        if ctx.needs_input_grad[1]:
            dw = _wgrad(x_buf, cin, dv_buf, cout, kh, kw, pad)
        if has_res and ctx.needs_input_grad[3]:
            dres = dv_buf
        return dx, dw, db, dres, None, None, None, None, None, None, None


def conv(x_buf, w, bias=None, res_buf=None, act=ACT_NONE, out_fp32_nchw=False, pad=None, out_f32_nhwc=False, out_hw=None, gate_in=ACT_NONE,
         gated_out=False):
    pad = w.shape[2] // 2 if pad is None else pad
    return ConvFn.apply(x_buf, w, bias, res_buf, act, out_fp32_nchw, pad, out_f32_nhwc, out_hw, gate_in, gated_out)


class SpadeFn(torch.autograd.Function):
    """h = act(InstanceNorm(xs + noise*ns) * (1 + conv(actv,Wg)+bg) + conv(actv,Wb)+bb), xs = cat(up2^shift(x0), x1).
    Forward: hrv_instnorm_stats + hrv_conv2d_fwd (SPADE epilogue, which also emits gamma for the backward).
    Backward: hrv_norm_bwd_reduce / hrv_norm_bwd_apply (fused modulation + InstanceNorm backward), then the dgrad of the
    gamma|beta GEMM through hrv_conv2d_fwd and its weight gradient."""

    @staticmethod
    def forward(ctx, actv_buf, wg, wb, bg, bb, x0_buf, x1_buf, noise, ns, x0_shift, act, stats=None):
        n, h, w, _ = actv_buf.shape
        c0 = x0_buf.shape[3]
        c1 = x1_buf.shape[3] if x1_buf is not None else 0
        C = c0 + c1
        x0, x1 = Act(x0_buf), (Act(x1_buf) if x1_buf is not None else None)
        nsd = ns.detach().float().contiguous()
        mean, rstd = stats if stats is not None else ops.instnorm_stats2(x0, x0_shift, x1, h, w, [noise], [nsd])[0]
        gb = ops.pack_weight(wg.detach(), (1, 1), interleave=wb.detach())
        gb_bias = torch.stack([bg.detach(), bb.detach()], 1).reshape(-1).float().contiguous()
        out = Act.empty(n, h, w, C)
        gamma = Act.empty(n, h, w, C)
        ops.conv2d_spade(Act(actv_buf, c=wg.shape[1]), gb, out, x0, x0_shift, x1, mean, rstd, noise, nsd, gb_bias, act, gamma_out=gamma)
        ctx.save_for_backward(actv_buf, wg, wb, x0_buf, x1_buf, noise, nsd, mean, rstd, out.buf, gamma.buf)
        ctx.meta = (x0_shift, act)
        return out.buf

    @staticmethod
    def backward(ctx, dout):
        actv_buf, wg, wb, x0_buf, x1_buf, noise, nsd, mean, rstd, out, gamma = ctx.saved_tensors
        x0_shift, act = ctx.meta
        n, h, w, _ = actv_buf.shape
        C = x0_buf.shape[3] + (x1_buf.shape[3] if x1_buf is not None else 0)
        dgb, dx0, dx1, dns, sum_dg, sum_db = ops.norm_bwd(
            Act(dout.contiguous()), Act(out), Act(gamma), Act(x0_buf), x0_shift, Act(x1_buf) if x1_buf is not None else None,
            noise, nsd, mean, rstd, act, want_dgb=True)
        dactv = None
        if ctx.needs_input_grad[0]:
            pw = ops.pack_weight(wg, (1, 1), interleave=wb, dgrad=True)  # K = interleaved (gamma_c, beta_c) columns of dgb
            da = Act.empty(n, h, w, wg.shape[1], pitch=actv_buf.shape[3], zero=actv_buf.shape[3] > wg.shape[1])
            ops.conv2d(dgb, pw, da)
            dactv = da.buf
        dwcat = _wgrad(actv_buf, wg.shape[1], dgb.buf, 2 * C, 3, 3, 1)
        return (dactv, dwcat[0::2].contiguous(), dwcat[1::2].contiguous(), sum_dg, sum_db,
                dx0.buf if ctx.needs_input_grad[5] else None,
                dx1.buf if (dx1 is not None and ctx.needs_input_grad[6]) else None, None, dns, None, None, None)


class FromNCHW(torch.autograd.Function):
    """fp32 NCHW -> pixel-major bf16 (with nearest resize); backward only when the input needs a gradient."""

    @staticmethod
    def forward(ctx, x, size, c_pad):
        ctx.shape = x.shape
        ctx.size = size
        return ops.from_nchw(x.float().contiguous(), c_pad=c_pad, size=size).buf

    @staticmethod
    def backward(ctx, dbuf):
        n, c, h, w = ctx.shape
        if ctx.size is not None and tuple(ctx.size) != (h, w):
            raise NotImplementedError("gradient through the nearest-resized input pyramid is never needed (inputs are data)")
        return Act(dbuf.contiguous(), c=c).to_nchw(), None, None


def _block_train(blk, x0_buf, x0_shift, x1_buf, seg_buf, noise_fn, out_act):
    """SPADEResBlock forward with autograd nodes (network_generator.py:157-173)."""
    n, h, w, _ = seg_buf.shape
    seg_c = blk.norm_0.conv_shared[0].weight.shape[1]
    # 3x3 over the few-channel label map: gather the 9 taps once per block (shared by its 2-3 norms) so each mlp_shared
    # convolution is a single K=64 GEMM block per pixel tile and its weight gradient a 1x1 GEMM
    cols = ops.im2col(Act(seg_buf, c=seg_c), 3, 3, 1).buf if 9 * seg_c <= 64 else None

    def spade(norm, x0b, sh, x1b, act, noise=None, stats=None):
        cs = norm.conv_shared[0]
        if cols is not None:
            actv = conv(cols, im2col_weight(cs.weight, cols.shape[3]), cs.bias, act=ACT_RELU, pad=0)
        else:
            actv = conv(seg_buf, cs.weight, cs.bias, act=ACT_RELU)
        return SpadeFn.apply(actv, norm.conv_gamma.weight, norm.conv_beta.weight, norm.conv_gamma.bias, norm.conv_beta.bias,
                             x0b, x1b, noise if noise is not None else noise_fn(n, h, w), norm.noise_scale, sh, act, stats)

    if blk.learned_shortcut:
        # norm_s and norm_0 share their input (own noise each): one statistics pass over the source tensors serves both
        nz_s, nz_0 = noise_fn(n, h, w), noise_fn(n, h, w)
        st_s, st_0 = ops.instnorm_stats2(Act(x0_buf), x0_shift, Act(x1_buf) if x1_buf is not None else None, h, w, [nz_s, nz_0],
                                         [blk.norm_s.noise_scale.detach().float().contiguous(), blk.norm_0.noise_scale.detach().float().contiguous()])
        hs = spade(blk.norm_s, x0_buf, x0_shift, x1_buf, ACT_NONE, nz_s, st_s)
        x_s = conv(hs, conv_weight(blk.conv_s, blk.training))
        h0 = spade(blk.norm_0, x0_buf, x0_shift, x1_buf, ACT_LRELU, nz_0, st_0)
    else:
        x_s = x0_buf
        h0 = spade(blk.norm_0, x0_buf, x0_shift, x1_buf, ACT_LRELU)
    dx = conv(h0, conv_weight(blk.conv_0, blk.training), blk.conv_0.bias)
    h1 = spade(blk.norm_1, dx, 0, None, ACT_LRELU)
    return conv(h1, conv_weight(blk.conv_1, blk.training), blk.conv_1.bias, res_buf=x_s, act=out_act)


def generator_forward_train(g, x, seg):
    """SPADEGenerator.forward with a differentiable graph (network_generator.py:221-245)."""
    dev = x.device
    noise_fn = g.noise_source or (lambda b, hh, ww: torch.randn(b, hh, ww, device=dev))
    sizes = [(g.sh * 2 ** i, g.sw * 2 ** i) for i in range(8)]
    x = x.float()
    seg = seg.float()
    feats, segs = [], []
    for i, sz in enumerate(sizes):
        s = FromNCHW.apply(x, sz, 16)
        c = getattr(g, "conv_%d" % i)
        feats.append(conv(s, c.weight, c.bias))
        segs.append(ops.from_nchw(seg.detach(), size=sz).buf)
    h = _block_train(g.head_0, feats[0], 0, None, segs[0], noise_fn, ACT_NONE)
    names = g._blocks[1:]
    for j, name in enumerate(names):
        last = j == len(names) - 1
        h = _block_train(getattr(g, name), h, 1, feats[j + 1], segs[j + 1], noise_fn, ACT_LRELU if last else ACT_NONE)
    return conv(h, g.conv_img.weight, g.conv_img.bias, act=ACT_TANH, out_fp32_nchw=True)


# ------------------------------------------------------------------------------------------------ discriminator

class S2DFn(torch.autograd.Function):
    """Space-to-depth by 2 with zero fill of odd edges, channel order (py*2+px)*C8 + c (hrv_space_to_depth / ops.s2d_weight
    convention) and its inverse gather as the backward: one kernel each way, no pad / permute copies."""

    @staticmethod
    def forward(ctx, x_buf, cin):
        ctx.meta = (x_buf.shape, cin)
        return ops.space_to_depth(Act(x_buf, c=cin)).buf

    @staticmethod
    def backward(ctx, d):
        (n, h, w, p), cin = ctx.meta
        dx = ops.space_to_depth_bwd(Act(d.contiguous()), n, h, w, cin, pitch=p)
        if p > ops.round_up(cin, 8):
            dx.buf[..., ops.round_up(cin, 8):] = 0
        return dx.buf, None


def space_to_depth_t(x_buf, cin=None):
    return S2DFn.apply(x_buf, x_buf.shape[3] if cin is None else cin)


class MaxPool2Fn(torch.autograd.Function):
    """nn.MaxPool2d(2,2) on a pixel-major bf16 buffer (Vgg19, networks.py:201-231): hrv_maxpool2_fwd / hrv_maxpool2_bwd."""

    @staticmethod
    def forward(ctx, x_buf, relu_gate=False):
        ctx.save_for_backward(x_buf)
        ctx.relu_gate = relu_gate  # x_buf is a ReLU output whose producer expects dL/dv: apply (x > 0) while routing
        return ops.maxpool2(Act(x_buf)).buf

    @staticmethod
    def backward(ctx, dy):
        (x_buf,) = ctx.saved_tensors
        return ops.maxpool2_bwd(Act(x_buf), Act(dy.contiguous()), relu_gate=ctx.relu_gate).buf, None


class AvgPool3S2Fn(torch.autograd.Function):
    """F.avg_pool2d(3, stride 2, padding 1, count_include_pad=False) between discriminator scales (network_generator.py:302)
    on the pixel-major bf16 buffer: hrv_avgpool3s2 / hrv_avgpool3s2_bwd."""

    @staticmethod
    def forward(ctx, x_buf):
        ctx.hw = x_buf.shape[1:3]
        return ops.avgpool3s2(Act(x_buf)).buf

    @staticmethod
    def backward(ctx, dy):
        return ops.avgpool3s2_bwd(Act(dy.contiguous()), *ctx.hw).buf


class InstNormActFn(torch.autograd.Function):
    """y = act(InstanceNorm(x)) on a pixel-major bf16 buffer (network_generator.py:427 + LeakyReLU); backward through the
    same fused kernels as the SPADE norms (no modulation, no noise)."""

    @staticmethod
    def forward(ctx, x_buf, act):
        a = Act(x_buf)
        mean, rstd = ops.instnorm_stats(a, 0, None, a.h, a.w, None, None)
        y = Act.empty(a.n, a.h, a.w, a.c)
        ops.instnorm_apply(a, mean, rstd, act, out=y)
        ctx.save_for_backward(x_buf, mean, rstd, y.buf)
        ctx.act = act
        return y.buf

    @staticmethod
    def backward(ctx, dy):
        x_buf, mean, rstd, y = ctx.saved_tensors
        _, dx, _, _, _, _ = ops.norm_bwd(Act(dy.contiguous()), Act(y), None, Act(x_buf), 0, None, None, None, mean, rstd, ctx.act,
                                         want_dgb=False)
        return dx.buf, None


def patchgan_forward(seqs, x_buf, training, need_wgrad=True):
    """PatchGAN discriminator layers (network_generator.py:250-291, networks.py:351-408) on a pixel-major input.  Each nn.Sequential
    (nested ones flattened) chains Conv2d 4x4 (stride 2 | 1, pad 2), each followed by an optional InstanceNorm2d, an optional LeakyReLU
    and an optional Dropout, and runs on the previous one's output.  Returns each sequence's output buffer (fp32 for the 1-channel
    last layer).  need_wgrad=False detaches the weights (D inside the G step)."""
    outs = []
    h = x_buf
    for seq in seqs:
        mods = [m for m in seq.modules() if not isinstance(m, torch.nn.Sequential)]
        j = 0
        while j < len(mods):
            m = mods[j]
            if isinstance(m, torch.nn.Conv2d):
                nxt = mods[j + 1:j + 3]
                if nxt and isinstance(nxt[0], torch.nn.BatchNorm2d):
                    raise NotImplementedError("BatchNorm discriminators have no kernel (the reference uses norm='instance')")
                has_in = bool(nxt) and isinstance(nxt[0], torch.nn.InstanceNorm2d)
                has_lr = len(nxt) > has_in and isinstance(nxt[has_in], torch.nn.LeakyReLU)
                w, bias = conv_weight(m, training), m.bias
                if not need_wgrad:
                    w, bias = w.detach(), (bias.detach() if bias is not None else None)
                act = ACT_LRELU if (has_lr and not has_in) else ACT_NONE
                if m.stride[0] == 2:
                    # k4 s2 p2 on (H,W) == k2 s1 p1 on the space-to-depth tensor; extent floor(H/2)+1 (one less than the s2d conv's
                    # natural extent when H is odd: the kernels simply do not compute / read the cropped row)
                    y = conv(space_to_depth_t(h, w.shape[1]), ops.s2d_weight(w, 2), bias, act=act, pad=1,
                             out_hw=(h.shape[1] // 2 + 1, h.shape[2] // 2 + 1))
                else:
                    y = conv(h, w, bias, act=act, pad=2, out_f32_nhwc=w.shape[0] == 1)
                h = InstNormActFn.apply(y, ACT_LRELU if has_lr else ACT_NONE) if has_in else y
                j += 1 + has_in + has_lr
            elif isinstance(m, torch.nn.Dropout):
                h = F.dropout(h, m.p, training)
                j += 1
            elif isinstance(m, torch.nn.Sigmoid):
                raise NotImplementedError("use_sigmoid=True has no kernel (the reference uses LSGAN, use_sigmoid=False)")
            else:
                raise NotImplementedError("unexpected layer %s in a PatchGAN sequence" % type(m).__name__)
        outs.append(h)
    return outs


def nchw(buf, as_float=True):
    """NCHW form of a pixel-major output: while autograd records, the differentiable permuted view (fp32 when as_float); otherwise a
    contiguous fp32 copy (hrv_nhwc_to_nchw)."""
    if not torch.is_grad_enabled():
        return Act(buf).to_nchw()
    v = buf.permute(0, 3, 1, 2)
    return v.float() if as_float else v


class FeatMatchFn(torch.autograd.Function):
    """One term of the GAN feature-matching loss (train_generator.py:303-311): mean |D_j(fake) - D_j(real).detach()| where the
    discriminator ran on the concatenation [fake; real] along the batch axis, so one pixel-major buffer holds both halves.  Forward =
    hrv_l1_sum over the two halves; backward = hrv_l1_bwd into the first half of a zeroed gradient buffer (the real half carries no
    gradient).  Replaces four strided torch element-wise passes (sub, abs, sgn*g, slice-backward copy) per feature map."""

    @staticmethod
    def forward(ctx, buf):
        half = buf.shape[0] // 2
        ctx.save_for_backward(buf)
        a, b = Act(buf[:half]), Act(buf[half:])
        return (ops.l1_sum(a, b) / float(a.n * a.h * a.w * a.c)).float().reshape(())

    @staticmethod
    def backward(ctx, g):
        (buf,) = ctx.saved_tensors
        half = buf.shape[0] // 2
        a, b = Act(buf[:half]), Act(buf[half:])
        d = torch.empty_like(buf)
        d[half:].zero_()
        gscale = (g.float() / float(a.n * a.h * a.w * a.c)).reshape(1).contiguous()
        ops.l1_bwd(a, b, gscale, out=Act(d[:half]))
        return d


def discriminator_forward_train(D, input_nchw, need_wgrad=True, as_float=True, raw=False):
    """MultiscaleDiscriminator.forward (network_generator.py:293-316); returns NCHW feature lists (see nchw)
    (raw=True: the pixel-major buffers themselves for the intermediate features — FeatMatchFn's operand — and the NCHW view of the
    last, 1-channel output)."""
    cur = FromNCHW.apply(input_nchw, None, None)
    result = []
    ds = list(D.children())
    for k, d in enumerate(ds):
        outs = patchgan_forward(list(d.children()), cur, d.training, need_wgrad)
        feats = [o if raw and j + 1 < len(outs) else nchw(o, as_float) for j, o in enumerate(outs)]
        result.append(feats if not D.no_ganFeat_loss else [feats[-1]])
        if k + 1 < len(ds):
            cur = AvgPool3S2Fn.apply(cur)
    return result


# ------------------------------------------------------------------------------------------------ VGG19 feature loss

def vgg_features(vgg, x_nchw):
    """Vgg19.forward (networks.py:201-231) through the conv kernels: conv3x3+bias+ReLU fused, 2x2 max-pool as a torch
    data-movement op on the channels-last buffer.  Weights are frozen, so the backward is dgrad only (all ours).
    Returns the 5 slice outputs as pixel-major bf16 buffers."""
    h = FromNCHW.apply(x_nchw, None, None)
    outs = []
    relu_out = False  # is h the output of a conv+ReLU whose backward its consumers apply (gated_out)?
    for k in range(5):
        for layer in getattr(vgg, "slice%d" % (k + 1)):
            if isinstance(layer, torch.nn.Conv2d):
                # ReLU backward is never a pass of its own: the consumer of each activation (next convolution's data gradient,
                # max-pool backward, L1 backward) multiplies by (y > 0) in its epilogue
                h = conv(h, layer.weight, layer.bias, act=ACT_RELU, gate_in=ACT_RELU if relu_out else ACT_NONE, gated_out=True)
                relu_out = True
            elif isinstance(layer, torch.nn.MaxPool2d):
                h = MaxPool2Fn.apply(h, relu_out)
                relu_out = False
            elif isinstance(layer, torch.nn.ReLU):
                pass  # fused into the preceding convolution's epilogue
            else:
                raise NotImplementedError(type(layer).__name__)
        outs.append(h)
    return outs


class L1MeanFn(torch.autograd.Function):
    """mean |a - b| over two pixel-major bf16 buffers (b carries no gradient): hrv_l1_sum / hrv_l1_bwd, one pass each."""

    @staticmethod
    def forward(ctx, a_buf, b_buf, relu_gate=False):
        ctx.save_for_backward(a_buf, b_buf)
        ctx.relu_gate = relu_gate  # a_buf is a ReLU output whose producer expects dL/dv
        return (ops.l1_sum(Act(a_buf), Act(b_buf)) / a_buf.numel()).float().reshape(())

    @staticmethod
    def backward(ctx, g):
        a_buf, b_buf = ctx.saved_tensors
        gscale = (g.float() / a_buf.numel()).reshape(1).contiguous()
        return ops.l1_bwd(Act(a_buf), Act(b_buf), gscale, relu_gate=ctx.relu_gate).buf, None, None


def vgg_loss(vgg, weights, x, y):
    """VGGLoss.forward (networks.py:244-251): sum_i w_i * L1(vgg_i(x), vgg_i(y).detach())."""
    with torch.no_grad():  # the target branch carries no gradient: keep it out of the graph so the backward runs over x only
        fy = vgg_features(vgg, y.detach())
    fx = vgg_features(vgg, x)
    loss = 0
    for wgt, tx, ty in zip(weights, fx, fy):
        loss = loss + wgt * L1MeanFn.apply(tx, ty, True)  # every slice output is a conv+ReLU output with gated_out=True
    return loss
