"""Per-op gradient check of hrviton_b200.autograd_g nodes against torch autograd (fp32, same GPU)."""
import os, sys, torch
import torch.nn.functional as F
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hrv_loader; hrv_loader.load()
from hrviton_b200 import autograd_g as ag, ops
torch.manual_seed(0)
dev = "cuda"

def rel(a, b): return float((a.float() - b.float()).norm() / (b.float().norm() + 1e-12))

def check_conv(cin, cout, k, pad, h, w, f32_nhwc=False, act=0):
    x = torch.randn(2, cin, h, w, device=dev).bfloat16().float().requires_grad_(True)
    wt = (torch.randn(cout, cin, k, k, device=dev) * 0.1).bfloat16().float().requires_grad_(True)
    b = torch.randn(cout, device=dev).requires_grad_(True)
    y_ref = F.conv2d(x, wt, b, padding=pad)
    if act == 2: y_ref = F.leaky_relu(y_ref, 0.2)
    R = torch.randn_like(y_ref)
    (y_ref * R).sum().backward()
    gx, gw, gb = x.grad.clone(), wt.grad.clone(), b.grad.clone()
    x2 = x.detach().clone().requires_grad_(True); w2 = wt.detach().clone().requires_grad_(True); b2 = b.detach().clone().requires_grad_(True)
    xb = ag.FromNCHW.apply(x2, None, None)
    y = ag.conv(xb, w2, b2, act=act, pad=pad, out_f32_nhwc=f32_nhwc)
    yn = y[..., :cout].permute(0, 3, 1, 2).float()
    (yn * R).sum().backward()
    print("conv %d->%d k%d p%d %dx%d f32=%s act=%d: fwd %.2e dx %.2e dw %.2e db %.2e" % (cin, cout, k, pad, h, w, f32_nhwc, act, rel(yn, y_ref), rel(x2.grad, gx), rel(w2.grad, gw), rel(b2.grad, gb)))

check_conv(16, 32, 3, 1, 24, 16)
check_conv(64, 64, 2, 1, 17, 13, act=2)
check_conv(64, 1, 4, 2, 17, 13, f32_nhwc=True)
check_conv(10, 16, 3, 1, 16, 12)
# instnorm + lrelu
x = torch.randn(2, 32, 17, 13, device=dev).bfloat16().float().requires_grad_(True)
y_ref = F.leaky_relu(F.instance_norm(x), 0.2); R = torch.randn_like(y_ref); (y_ref * R).sum().backward()
x2 = x.detach().clone().requires_grad_(True)
y = ag.InstNormActFn.apply(ag.FromNCHW.apply(x2, None, None), 2)
yn = y.permute(0, 3, 1, 2).float(); (yn * R).sum().backward()
print("instnorm+lrelu: fwd %.2e dx %.2e" % (rel(yn, y_ref), rel(x2.grad, x.grad)))
# s2d conv k4 s2 p2
for (h, w) in [(16, 12), (17, 13)]:
    x = torch.randn(2, 10, h, w, device=dev).bfloat16().float().requires_grad_(True)
    wt = (torch.randn(24, 10, 4, 4, device=dev) * 0.1).bfloat16().float().requires_grad_(True)
    y_ref = F.conv2d(x, wt, None, stride=2, padding=2); R = torch.randn_like(y_ref); (y_ref * R).sum().backward()
    x2 = x.detach().clone().requires_grad_(True); w2 = wt.detach().clone().requires_grad_(True)
    src = ag.space_to_depth_t(ag.FromNCHW.apply(x2, None, None))
    y = ag.conv(src, ops.s2d_weight(w2, 2), None, pad=1)
    y = y[:, :y_ref.shape[2], :y_ref.shape[3], :24].permute(0, 3, 1, 2).float()
    (y * R).sum().backward()
    print("s2d conv %dx%d: fwd %.2e dx %.2e dw %.2e" % (h, w, rel(y, y_ref), rel(x2.grad, x.grad), rel(w2.grad, wt.grad)))
# ---- train-mode BatchNorm + ReLU (+ residual), c = 13 (padded) and 96
from hrviton_b200 import autograd_tocg as at
for c, with_res in [(96, True), (13, True), (96, False)]:
    bn = torch.nn.BatchNorm2d(c).to(dev).train()
    with torch.no_grad():
        bn.weight.uniform_(0.5, 1.5); bn.bias.normal_(0, 0.2)
    x = torch.randn(2, c, 17, 13, device=dev).bfloat16().float().requires_grad_(True)
    r = torch.randn(2, c, 17, 13, device=dev).bfloat16().float().requires_grad_(True)
    y_ref = torch.relu(bn(x) + (r if with_res else 0)); R = torch.randn_like(y_ref); (y_ref * R).sum().backward()
    gx, gr, gw, gb = x.grad.clone(), (r.grad.clone() if with_res else None), bn.weight.grad.clone(), bn.bias.grad.clone()
    rm_ref = bn.running_mean.clone(); rv_ref = bn.running_var.clone()
    bn2 = torch.nn.BatchNorm2d(c).to(dev).train()
    with torch.no_grad():
        bn2.weight.copy_(bn.weight); bn2.bias.copy_(bn.bias)
    x2 = x.detach().clone().requires_grad_(True); r2 = r.detach().clone().requires_grad_(True)
    y = at.BatchNormActFn.apply(ag.FromNCHW.apply(x2, None, None), bn2.weight, bn2.bias, ag.FromNCHW.apply(r2, None, None) if with_res else None, bn2, 1)
    yn = y[..., :c].permute(0, 3, 1, 2).float(); (yn * R).sum().backward()
    print("bn_train c=%d res=%s: fwd %.2e dx %.2e dres %s dw %.2e db %.2e  run_mean %.2e run_var %.2e" % (
        c, with_res, rel(yn, y_ref), rel(x2.grad, gx), ("%.2e" % rel(r2.grad, gr)) if with_res else "-", rel(bn2.weight.grad, gw), rel(bn2.bias.grad, gb),
        rel(bn2.running_mean, rm_ref), rel(bn2.running_var, rv_ref)))
# ---- 3x3 stride-2 pad-1 conv through space-to-depth
for (h, w) in [(16, 12), (17, 13)]:
    x = torch.randn(2, 4, h, w, device=dev).bfloat16().float().requires_grad_(True)
    wt = (torch.randn(24, 4, 3, 3, device=dev) * 0.1).bfloat16().float().requires_grad_(True)
    y_ref = F.conv2d(x, wt, None, stride=2, padding=1); R = torch.randn_like(y_ref); (y_ref * R).sum().backward()
    x2 = x.detach().clone().requires_grad_(True); w2 = wt.detach().clone().requires_grad_(True)
    src = ag.space_to_depth_t(ag.FromNCHW.apply(x2, None, None))
    y = ag.conv(src, ops.s2d_weight(w2, 1), None, pad=1)
    y = y[:, :y_ref.shape[2], :y_ref.shape[3], :24].permute(0, 3, 1, 2).float()
    (y * R).sum().backward()
    print("s2d conv k3s2p1 %dx%d: fwd %.2e dx %.2e dw %.2e" % (h, w, rel(y, y_ref), rel(x2.grad, x.grad), rel(w2.grad, wt.grad)))
# ---- bilinear x2 (+add) and the fused flow warp: kernel forward/backward vs torch autograd
def warp_ref(src_nchw, flow_lo):
    """networks.py:133-135 / 147-152 in torch: flow x2 (bilinear), normalise by ((W/2-1)/2,(H/2-1)/2), + base grid, grid_sample(border)."""
    n, _, h, w = src_nchw.shape
    fl = F.interpolate(flow_lo.permute(0, 3, 1, 2), scale_factor=2, mode="bilinear", align_corners=False).permute(0, 2, 3, 1)
    fn = torch.cat([fl[..., 0:1] / ((w / 2 - 1.0) / 2.0), fl[..., 1:2] / ((h / 2 - 1.0) / 2.0)], 3)
    gx = torch.linspace(-1.0, 1.0, w).view(1, 1, w, 1).expand(n, h, w, 1)
    gy = torch.linspace(-1.0, 1.0, h).view(1, h, 1, 1).expand(n, h, w, 1)
    grid = torch.cat([gx, gy], 3).to(src_nchw.device)
    return F.grid_sample(src_nchw, fn + grid, mode="bilinear", padding_mode="border", align_corners=False), fl
a = torch.randn(2, 24, 9, 7, device=dev).bfloat16().float().requires_grad_(True)
b = torch.randn(2, 24, 18, 14, device=dev).bfloat16().float().requires_grad_(True)
y_ref = F.interpolate(a, scale_factor=2, mode="bilinear", align_corners=False) + b; R = torch.randn_like(y_ref); (y_ref * R).sum().backward()
a2 = a.detach().clone().requires_grad_(True); b2 = b.detach().clone().requires_grad_(True)
y = at.Up2Fn.apply(ag.FromNCHW.apply(a2, None, None), ag.FromNCHW.apply(b2, None, None)); yn = y.permute(0, 3, 1, 2).float(); (yn * R).sum().backward()
print("up2_add: fwd %.2e da %.2e db %.2e" % (rel(yn, y_ref), rel(a2.grad, a.grad), rel(b2.grad, b.grad)))
for c in (48, 4):
    src = torch.randn(2, c, 32, 24, device=dev).bfloat16().float().requires_grad_(True)
    flow = (torch.randn(2, 16, 12, 2, device=dev) * 2.5).requires_grad_(True)
    w_ref, fu_ref = warp_ref(src, flow); R = torch.randn_like(w_ref); R2 = torch.randn_like(fu_ref)
    ((w_ref * R).sum() + (fu_ref * R2).sum()).backward()
    s2 = src.detach().clone().requires_grad_(True); f2 = flow.detach().clone().requires_grad_(True)
    wb, fu = at.FlowWarpFn.apply(ag.FromNCHW.apply(s2, None, None), f2)
    wn = wb[..., :c].permute(0, 3, 1, 2).float()
    ((wn * R).sum() + (fu * R2).sum()).backward()
    print("flow_warp c=%d: fwd %.2e flow_up %.2e dsrc %.2e dflow %.2e" % (c, rel(wn, w_ref), rel(fu, fu_ref), rel(s2.grad, src.grad), rel(f2.grad, flow.grad)))
