"""Training path (forward + backward) of the condition generator ("tocg") and the stage-1 discriminator.

Convolutions (forward, dgrad, wgrad), train-mode BatchNorm (single-pass batch statistics + fused normalise/affine/ReLU/residual,
fused backward), InstanceNorm and activations run on this repo's kernels through the autograd nodes of autograd_g.  The resampling between them is on kernels too: bilinear x2 (+ lateral add) forward/backward (hrv_bilinear_up2_add / _bwd)
and the fused appearance-flow warp forward/backward (hrv_flow_warp / hrv_flow_warp_bwd).  Only channel concatenations (torch.cat) and the
dropout of the stage-1 discriminator remain torch ops in this training path."""
import torch
import torch.nn.functional as F

from . import ops
from .autograd_g import AvgPool3S2Fn, FromNCHW, conv, nchw, patchgan_forward, space_to_depth_t
from .ops import ACT_RELU, Act


class BatchNormActFn(torch.autograd.Function):
    """y = act(BatchNorm2d_train(x) (+ res)) on a pixel-major bf16 buffer (networks.py:188-198): batch statistics from one pass of the
    statistics kernel, running statistics updated as torch's BatchNorm2d does (momentum, unbiased variance)."""

    @staticmethod
    def forward(ctx, x_buf, weight, bias, res_buf, bn, act):
        c = weight.shape[0]
        c8 = ops.round_up(c, 8)  # kernels work on groups of 8 channels; pad channels hold zeros and get weight = bias = 0
        a = Act(x_buf, c=c8)
        n = a.n
        mean, var = ops.batchnorm_stats(a, bn.eps)
        if bn.track_running_stats and bn.training:
            with torch.no_grad():
                cnt = float(n * a.h * a.w)
                m = bn.momentum if bn.momentum is not None else 0.1
                bn.running_mean.mul_(1 - m).add_(mean[:c] * m)
                bn.running_var.mul_(1 - m).add_(var[:c] * (cnt / max(cnt - 1.0, 1.0)) * m)
                bn.num_batches_tracked += 1
        rstd = torch.rsqrt(var + bn.eps)
        mean_nc = mean[None].expand(n, c8).contiguous()
        rstd_nc = rstd[None].expand(n, c8).contiguous()
        w32 = torch.zeros(c8, dtype=torch.float32, device=x_buf.device)
        b32 = torch.zeros(c8, dtype=torch.float32, device=x_buf.device)
        w32[:c] = weight.detach().float()
        b32[:c] = bias.detach().float()
        y = ops.norm_apply_affine(a, mean_nc, rstd_nc, w32, b32, Act(res_buf, c=c8) if res_buf is not None else None, act)
        ctx.save_for_backward(x_buf, w32, mean_nc, rstd_nc, y.buf)
        ctx.meta = (act, res_buf is not None, c, c8)
        return y.buf

    @staticmethod
    def backward(ctx, dy):
        x_buf, w32, mean_nc, rstd_nc, y = ctx.saved_tensors
        act, has_res, c, c8 = ctx.meta
        dya = Act(dy.contiguous(), c=c8)
        _, dx, _, _, dgamma, dbeta = ops.norm_bwd(dya, Act(y, c=c8), None, Act(x_buf, c=c8), 0, None, None, None, mean_nc, rstd_nc, act,
                                                  want_dgb=False, chan_scale=w32, batch_stats=True)
        dres = None
        if has_res and ctx.needs_input_grad[3]:
            dres = ops.act_bwd_bias(dya, Act(y, c=c8), act, want_bias=False)[0].buf
        dxb = dx.buf
        if dxb.shape[3] != x_buf.shape[3]:
            dxb = F.pad(dxb, (0, x_buf.shape[3] - dxb.shape[3]))
        return dxb, dgamma[:c].contiguous(), dbeta[:c].contiguous(), dres, None, None


class Up2Fn(torch.autograd.Function):
    """out = bilinear_up2(a) (+ b) on pixel-major bf16 buffers (F.interpolate(x2, bilinear) [+ lateral], networks.py:130,181):
    hrv_bilinear_up2_add forward, hrv_bilinear_up2_bwd (adjoint gather) backward."""

    @staticmethod
    def forward(ctx, a_buf, b_buf):
        a = Act(a_buf)
        out = Act.empty(a.n, 2 * a.h, 2 * a.w, a.c, pitch=a_buf.shape[3])
        ops.bilinear_up2_add(a, Act(b_buf) if b_buf is not None else None, out)
        return out.buf

    @staticmethod
    def backward(ctx, dout):
        dout = dout.contiguous()
        da = ops.bilinear_up2_bwd(Act(dout)).buf if ctx.needs_input_grad[0] else None
        return da, (dout if ctx.needs_input_grad[1] else None)


def _up2(buf, add=None):
    return Up2Fn.apply(buf, add)


class FlowWarpFn(torch.autograd.Function):
    """(warped, flow_up) = hrv_flow_warp(src, flow_lo) — flow x2 bilinear + normalise + base grid + grid_sample(border) in one kernel
    (networks.py:133-135,147-152); backward = hrv_flow_warp_bwd (scatter-add d_src, analytic d_flow, adjoint of the flow up-sampling)."""

    @staticmethod
    def forward(ctx, src_buf, flow_lo):
        src = Act(src_buf)
        flow_lo = flow_lo.contiguous()
        dst = Act.empty(src.n, src.h, src.w, src.c, pitch=src_buf.shape[3])
        flow_up, _ = ops.flow_warp(flow_lo, src, dst)
        ctx.save_for_backward(src_buf, flow_lo)
        return dst.buf, flow_up

    @staticmethod
    def backward(ctx, d_dst, d_flow_up):
        src_buf, flow_lo = ctx.saved_tensors
        if d_dst is None:
            d_dst = torch.zeros_like(src_buf)
        dsrc, dflo = ops.flow_warp_bwd(flow_lo, Act(src_buf), Act(d_dst.contiguous()), d_flow_up, want_dsrc=ctx.needs_input_grad[0])
        return (dsrc.buf if dsrc is not None else None), dflo


def _resblock(rb, x_buf):
    """ResBlock.forward in training mode (networks.py:171-198)."""
    if rb.kind == "down":
        w = rb.scale.weight
        src = space_to_depth_t(x_buf, w.shape[1])
        oh, ow = (x_buf.shape[1] - 1) // 2 + 1, (x_buf.shape[2] - 1) // 2 + 1  # k3 s2 p1 extent; the s2d form would give one more
        r = conv(src, ops.s2d_weight(w, 1), rb.scale.bias, pad=1, out_hw=(oh, ow))
    elif rb.kind == "same":
        r = conv(x_buf, rb.scale.weight, rb.scale.bias, pad=0)
    else:
        r = _up2(conv(x_buf, rb.scale[1].weight, rb.scale[1].bias, pad=0))  # 1x1 commuted below the up-sampling (kernel fwd + bwd)
    bn0, bn1 = rb.block[1], rb.block[4]
    h = BatchNormActFn.apply(conv(r, rb.block[0].weight, rb.block[0].bias), bn0.weight, bn0.bias, None, bn0, ACT_RELU)
    return BatchNormActFn.apply(conv(h, rb.block[3].weight, rb.block[3].bias), bn1.weight, bn1.bias, r, bn1, ACT_RELU)


def tocg_forward_train(m, input1, input2):
    """ConditionGenerator.forward with a differentiable graph (networks.py:98-159), train-mode BatchNorm."""
    ngf = m.ngf
    a = FromNCHW.apply(input1.float(), None, None)
    b = FromNCHW.apply(input2.float(), None, None)
    a1, a2 = a, b
    e1, e2 = [], []
    for k in range(5):
        a = _resblock(m.ClothEncoder[k], a)
        b = _resblock(m.PoseEncoder[k], b)
        e1.append(a)
        e2.append(b)
    flows = []
    fc = m.flow_conv
    flow = conv(torch.cat([e1[4], e2[4]], 3), fc[0].weight, fc[0].bias, out_f32_nhwc=True)
    flows.append(flow)
    x = _resblock(m.SegDecoder[0], _resblock(m.conv, e2[4]))
    t1 = e1[4]
    for i in range(1, 5):
        lvl = 4 - i
        t1 = _up2(t1, conv(e1[lvl], m.conv1[lvl].weight, m.conv1[lvl].bias, pad=0))
        warped, flow_up = FlowWarpFn.apply(t1, flows[-1])
        bt = m.bottleneck[i - 1][0]
        bott = conv(x, bt.weight, bt.bias, act=ACT_RELU)
        flow = flow_up + conv(torch.cat([warped, bott], 3), fc[i].weight, fc[i].bias, out_f32_nhwc=True)
        flows.append(flow)
        x = _resblock(m.SegDecoder[i], torch.cat([x, e2[lvl], warped], 3))
    warped_in_buf, _ = FlowWarpFn.apply(a1, flows[-1])
    fin = torch.cat([x, a2, warped_in_buf], 3)
    seg_buf = _resblock(m.out_layer, fin)
    seg = seg_buf[..., :m.io[2]].permute(0, 3, 1, 2).float()
    c1 = m.io[0]
    warped_in = warped_in_buf[..., :c1].permute(0, 3, 1, 2).float()
    return flows, seg, warped_in[:, :-1], warped_in[:, -1:]


# ------------------------------------------------------------------------------------------------ stage-1 discriminator

def tocg_discriminator_forward_train(D, input_nchw):
    """networks.MultiscaleDiscriminator.forward (networks.py:331-349): list[num_D] of NCHW fp32 feature lists (see autograd_g.nchw), the
    per-layer features with getIntermFeat, else [logits]."""
    buf = FromNCHW.apply(input_nchw.float(), None, None)
    if D.Ddownx2:
        buf = AvgPool3S2Fn.apply(buf)
    res = []
    for i in range(D.num_D):
        k = D.num_D - 1 - i
        if D.getIntermFeat:
            seqs = [getattr(D, "scale%d_layer%d" % (k, j)) for j in range(D.n_layers + 2)]
        else:
            seqs = [getattr(D, "layer%d" % k)]
        res.append([nchw(o) for o in patchgan_forward(seqs, buf, D.training)])
        if i != D.num_D - 1:
            buf = AvgPool3S2Fn.apply(buf)
    return res
