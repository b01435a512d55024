"""GPU parity tests of every C-ABI kernel against CPU restatements (torch-CPU fp32 conv substrate and the
numpy index formulas of oracle/hrviton_oracle.py).  All calls go through the C-ABI (hrviton_b200.ops -> ctypes)."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "oracle"))
import hrviton_oracle as orc  # noqa: E402
from hrviton_b200 import capi, ops, synth  # noqa: E402
from hrviton_b200.ops import Act  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda"


def bf16r(t):
    return t.to(torch.bfloat16).float()


def rel_err(got, ref):
    got = got.detach().float().cpu()
    ref = ref.detach().float().cpu()
    assert got.shape == ref.shape, (got.shape, ref.shape)
    return float((got - ref).abs().max() / (ref.abs().max() + 1e-6))


def run_conv(n, cin, cout, h, w, k, pad, *, act=0, bias=True, scale=False, res=False, seed=0, out_fp32_nchw=False,
             in_pitch=None, stride=1):
    x = bf16r(synth.normalish((n, cin, h, w), seed, "x"))
    wt = bf16r(synth.normalish((cout, cin, k, k), seed, "w", (1.0 / (cin * k * k)) ** 0.5))
    b = synth.normalish((cout,), seed, "b", 0.1) if bias else None
    sc = synth.uniform((cout,), seed, "s", 0.5, 1.5) if scale else None
    ref = F.conv2d(x, wt, None, stride=stride, padding=pad)
    if sc is not None:
        ref = ref * sc[None, :, None, None]
    if b is not None:
        ref = ref + b[None, :, None, None]
    oh, ow = ref.shape[2:]
    r = bf16r(synth.normalish((n, cout, oh, ow), seed, "r")) if res else None
    if r is not None:
        ref = ref + r
    ref = {0: lambda t: t, 1: torch.relu, 2: lambda t: F.leaky_relu(t, 0.2), 3: torch.tanh}[act](ref)

    xa = ops.from_nchw(x.to(DEV), c_pad=in_pitch)
    if stride == 2:
        xa = ops.space_to_depth(xa)
        pw = ops.pack_weight(ops.s2d_weight(wt.to(DEV), pad), (1, 1), cin_total=xa.c)
    else:
        pw = ops.pack_weight(wt.to(DEV), (pad, pad))
    ra = ops.from_nchw(r.to(DEV)) if r is not None else None
    dsc = sc.to(DEV) if sc is not None else None
    dsh = b.to(DEV) if b is not None else None
    if out_fp32_nchw:
        out = torch.empty((n, cout, oh, ow), dtype=torch.float32, device=DEV)
        ops.conv2d(xa, pw, out, act=act, scale=dsc, shift=dsh, res=ra, out_layout=capi.NCHW)
        got = out
    else:
        oa = Act.empty(n, oh, ow, cout, zero=True)
        ops.conv2d(xa, pw, oa, act=act, scale=dsc, shift=dsh, res=ra)
        got = oa.to_nchw()
    torch.cuda.synchronize()
    return rel_err(got, ref)


CONV_CASES = [
    # n, cin, cout, h, w, k, pad, kwargs
    (2, 64, 64, 16, 16, 3, 1, {}),
    (1, 128, 160, 32, 24, 3, 1, dict(act=2)),
    (1, 80, 32, 64, 48, 3, 1, {}),
    (2, 7, 128, 32, 24, 3, 1, dict(act=1)),
    (1, 9, 16, 16, 12, 3, 1, {}),
    (2, 96, 384, 16, 12, 1, 0, {}),
    (3, 1040, 1024, 8, 6, 3, 1, {}),
    (1, 256, 1, 17, 13, 4, 2, dict(out_fp32_nchw=True)),
    (2, 10, 64, 33, 25, 4, 2, dict(stride=2, act=2)),
    (2, 64, 128, 33, 25, 4, 2, dict(stride=2, bias=False)),
    (1, 16, 96, 64, 48, 3, 1, dict(stride=2, bias=False)),
    (1, 4, 96, 32, 24, 3, 1, dict(stride=2, bias=False)),
    (2, 96, 96, 32, 24, 3, 1, dict(act=1, scale=True, res=True)),
    (1, 32, 3, 64, 48, 3, 1, dict(act=3, out_fp32_nchw=True)),
    (1, 768, 2, 16, 12, 3, 1, dict(out_fp32_nchw=True)),
    (2, 128, 160, 256, 192, 3, 1, dict(act=2)),  # 768 tiles: persistent loop, phase wrap, TMEM double buffering
    (1, 144, 64, 128, 96, 3, 1, {}),
]


@pytest.mark.parametrize("case", CONV_CASES, ids=lambda c: "n%d_%dto%d_%dx%d_k%dp%d_%s" % (c[0], c[1], c[2], c[3], c[4], c[5], c[6], "_".join("%s%s" % kv for kv in c[7].items())))
def test_conv(case):
    n, cin, cout, h, w, k, pad, kw = case
    err = run_conv(n, cin, cout, h, w, k, pad, **kw)
    print('conv rel err', case, err)
    assert err < 1e-2, err


def test_conv_channel_slices():
    """Input read through a channel-slice view (pitch > c), output written into a slice of a wider buffer
    (this is how torch.cat is eliminated)."""
    n, h, w = 1, 16, 12
    x = bf16r(synth.normalish((n, 96, h, w), 3, "x"))
    wt = bf16r(synth.normalish((64, 32, 3, 3), 3, "w", 0.06))
    ref = F.conv2d(x[:, 32:64], wt, None, padding=1)
    xa = ops.from_nchw(x.to(DEV))
    big = Act.empty(n, h, w, 128, zero=True)
    ops.conv2d(xa.slice(32, 32), ops.pack_weight(wt.to(DEV), (1, 1)), big.slice(64, 64))
    got = big.to_nchw()
    torch.cuda.synchronize()
    assert rel_err(got[:, 64:], ref) < 1e-2
    assert float(got[:, :64].abs().max()) == 0.0


@pytest.mark.parametrize("shift,with_x1,cx0", [(0, False, 64), (1, True, 64), (1, True, 1024), (0, True, 32)])
def test_conv_spade(shift, with_x1, cx0):
    n, h, w = 2, 32, 24
    if cx0 == 1024:
        n, h, w = 1, 16, 12
    cx1 = 16 if with_x1 else 0
    C = cx0 + cx1
    seed = 5
    actv = bf16r(synth.normalish((n, 128, h, w), seed, "actv").abs())
    wg = bf16r(synth.normalish((C, 128, 3, 3), seed, "wg", 0.03))
    wb = bf16r(synth.normalish((C, 128, 3, 3), seed, "wb", 0.03))
    bg = synth.normalish((C,), seed, "bg", 0.1)
    bb = synth.normalish((C,), seed, "bb", 0.1)
    x0 = bf16r(synth.normalish((n, cx0, h >> shift, w >> shift), seed, "x0"))
    x1 = bf16r(synth.normalish((n, cx1, h, w), seed, "x1")) if with_x1 else None
    noise = synth.spade_noise(n, h, w, seed, 0)
    ns = synth.normalish((C,), seed, "ns", 0.1)
    xs = F.interpolate(x0, scale_factor=2, mode="nearest") if shift else x0
    if x1 is not None:
        xs = torch.cat([xs, x1], 1)
    xn = xs + noise[:, None] * ns[None, :, None, None]
    m = xn.mean((2, 3), keepdim=True)
    v = xn.var((2, 3), unbiased=False, keepdim=True)
    normalized = (xn - m) / torch.sqrt(v + 1e-5)
    gamma = F.conv2d(actv, wg, bg, padding=1)
    beta = F.conv2d(actv, wb, bb, padding=1)
    ref = F.leaky_relu(normalized * (1 + gamma) + beta, 0.2)

    a_actv = ops.from_nchw(actv.to(DEV))
    a_x0 = ops.from_nchw(x0.to(DEV))
    a_x1 = ops.from_nchw(x1.to(DEV)) if x1 is not None else None
    d_noise, d_ns = noise.to(DEV).contiguous(), ns.to(DEV)
    mean, rstd = ops.instnorm_stats(a_x0, shift, a_x1, h, w, d_noise, d_ns)
    torch.cuda.synchronize()
    assert rel_err(mean, m[:, :, 0, 0]) < 2e-3 or float((mean.cpu() - m[:, :, 0, 0]).abs().max()) < 2e-3
    assert rel_err(rstd, 1.0 / torch.sqrt(v + 1e-5)[:, :, 0, 0]) < 2e-3
    pw = ops.pack_weight(wg.to(DEV), (1, 1), interleave=wb.to(DEV))
    shift_vec = torch.stack([bg, bb], 1).reshape(-1).to(DEV)
    out = Act.empty(n, h, w, C, zero=True)
    ops.conv2d_spade(a_actv, pw, out, a_x0, shift, a_x1, mean, rstd, d_noise, d_ns, shift_vec, ops.ACT_LRELU)
    got = out.to_nchw()
    torch.cuda.synchronize()
    assert rel_err(got, ref) < 1.5e-2


def test_instnorm_apply():
    x = bf16r(synth.normalish((2, 128, 17, 13), 7, "x", 2.0, 0.3))
    ref = F.leaky_relu(F.instance_norm(x, eps=1e-5), 0.2)
    a = ops.from_nchw(x.to(DEV))
    mean, rstd = ops.instnorm_stats(a, 0, None, 17, 13, None, None)
    ops.instnorm_apply(a, mean, rstd, ops.ACT_LRELU)
    assert rel_err(a.to_nchw(), ref) < 1e-2


def test_layout_and_nearest():
    x = synth.uniform((2, 9, 32, 24), 8, "x")
    for size in [(32, 24), (16, 12), (8, 6), (2, 1), (4, 3)]:
        a = ops.from_nchw(x.to(DEV), size=size)
        ref = bf16r(F.interpolate(x, size=size, mode="nearest"))
        got = a.to_nchw()
        assert float((got.cpu() - ref).abs().max()) == 0.0
        assert float(a.buf[..., 9:].abs().max()) == 0.0


def test_space_to_depth_and_avgpool():
    x = bf16r(synth.uniform((2, 16, 17, 13), 9, "x"))
    a = ops.from_nchw(x.to(DEV))
    s = ops.space_to_depth(a).to_nchw().cpu()
    xp = F.pad(x, (0, 1, 0, 1))
    for py in range(2):
        for px in range(2):
            sub = py * 2 + px
            assert float((s[:, sub * 16:(sub + 1) * 16] - xp[:, :, py::2, px::2]).abs().max()) == 0.0
    p = ops.avgpool3s2(a).to_nchw()
    ref = F.avg_pool2d(x, 3, stride=2, padding=1, count_include_pad=False)
    assert rel_err(p, ref) < 1e-2
    assert rel_err(p, torch.from_numpy(orc.np_avgpool3s2(x.numpy()))) < 1e-2


def test_bilinear_up2_add():
    a = bf16r(synth.uniform((2, 24, 8, 6), 10, "a"))
    b = bf16r(synth.uniform((2, 24, 16, 12), 10, "b"))
    ref = torch.from_numpy(orc.np_bilinear_up2(a.numpy())) + b
    out = Act.empty(2, 16, 12, 24)
    ops.bilinear_up2_add(ops.from_nchw(a.to(DEV)), ops.from_nchw(b.to(DEV)), out)
    assert rel_err(out.to_nchw(), ref) < 1e-2


@pytest.mark.parametrize("c,src_fp32", [(384, False), (4, True), (8, False)])
def test_flow_warp_bit_exact(c, src_fp32):
    """Gather indices and the up-sampled flow must be BIT-EXACT against the numpy restatement; values within bf16."""
    n, h, w = 2, 32, 24
    flow = synth.normalish((n, h // 2, w // 2, 2), 12, "fl", 3.0)
    src = synth.uniform((n, c, h, w), 12, "src")
    src_used = src if src_fp32 else bf16r(src)
    x0, y0, tx, ty = orc.np_flow_warp_coords(flow.numpy(), h, w, h, w)
    ref = torch.from_numpy(orc.np_gather_bilinear(src_used.numpy(), x0, y0, tx, ty))
    ref_flow_up = np.moveaxis(orc.np_bilinear_up2(np.moveaxis(flow.numpy(), -1, 1)), 1, -1)
    if src_fp32:
        sa = Act(src.permute(0, 2, 3, 1).contiguous().to(DEV))
        dst = Act.empty(n, h, w, c, dtype=torch.float32, pitch=c)
    else:
        sa = ops.from_nchw(src.to(DEV))
        dst = Act.empty(n, h, w, c)
    flow_up, idx = ops.flow_warp(flow.to(DEV).contiguous(), sa, dst, want_idx=True)
    torch.cuda.synchronize()
    idx = idx.cpu().numpy()
    assert np.array_equal(idx[..., 0], x0) and np.array_equal(idx[..., 1], y0)
    assert np.array_equal(flow_up.cpu().numpy(), ref_flow_up)
    got = dst.to_nchw()
    assert rel_err(got, ref) < (1e-5 if src_fp32 else 1e-2)
    # and against the torch substrate the reference actually calls
    assert rel_err(got, orc.flow_warp(src_used, flow)) < (1e-4 if src_fp32 else 1e-2)


WGRAD_CASES = [(2, 64, 128, 24, 16, 3, 1), (1, 128, 160, 32, 24, 3, 1), (2, 80, 32, 64, 48, 3, 1), (1, 7, 128, 32, 24, 3, 1),
               (1, 1040, 512, 16, 12, 3, 1), (2, 96, 384, 16, 12, 1, 0), (2, 64, 24, 17, 13, 2, 1), (1, 256, 1, 17, 13, 4, 2),
               (1, 32, 3, 128, 96, 3, 1), (2, 128, 288, 130, 70, 3, 1)]


@pytest.mark.parametrize("case", WGRAD_CASES, ids=lambda c: "n%d_%dto%d_%dx%d_k%dp%d" % c)
def test_conv_wgrad(case):
    """hrv_conv2d_wgrad vs torch's fp32 weight gradient of the same (bf16-rounded) operands."""
    n, cin, cout, h, w, k, pad = case
    x = bf16r(synth.normalish((n, cin, h, w), 21, "x"))
    oh, ow = h + 2 * pad - k + 1, w + 2 * pad - k + 1
    dy = bf16r(synth.normalish((n, cout, oh, ow), 21, "dy"))
    ref = torch.nn.grad.conv2d_weight(x, (cout, cin, k, k), dy, stride=1, padding=pad)
    got = ops.conv2d_wgrad(ops.from_nchw(x.to(DEV)), ops.from_nchw(dy.to(DEV)), k, k, pad)
    torch.cuda.synchronize()
    err = rel_err(got, ref)
    print("wgrad rel err", case, err)
    assert err < 2e-3


# ------------------------------------------------------------------------------------------------ training-step glue kernels

def _to_buf(x_nchw, pitch=None):
    """fp32 NCHW (cpu) -> (N,H,W,P) bf16 cuda buffer with zero pad channels."""
    n, c, h, w = x_nchw.shape
    p = ops.round_up(c, 8) if pitch is None else pitch
    buf = torch.zeros((n, h, w, p), dtype=torch.bfloat16, device=DEV)
    buf[..., :c] = x_nchw.permute(0, 2, 3, 1).to(DEV).to(torch.bfloat16)
    return buf


@pytest.mark.parametrize("shape", [(2, 10, 13, 9), (1, 64, 8, 12), (3, 24, 7, 7)])
def test_space_to_depth_bwd_is_the_adjoint(shape):
    """<S(x), d> == <x, S^T(d)> for exactly representable values, plus the explicit index formula."""
    n, c, h, w = shape
    c8 = ops.round_up(c, 8)
    h2, w2 = (h + 1) // 2, (w + 1) // 2
    d = bf16r(synth.normalish((n, h2, w2, 4 * c8), 3, "d")).to(DEV).to(torch.bfloat16).contiguous()
    dx = ops.space_to_depth_bwd(Act(d), n, h, w, c).buf.float().cpu()
    dref = d.float().cpu().reshape(n, h2, w2, 2, 2, c8)
    for y in range(h):
        for x in range(w):
            assert torch.equal(dx[:, y, x, :c], dref[:, y // 2, x // 2, y & 1, x & 1, :c]), (y, x)
    # forward/backward pair consistency on a one-hot probe
    xb = _to_buf(bf16r(synth.normalish(shape, 4, "x")))
    s = ops.space_to_depth(Act(xb, c=c)).buf
    back = ops.space_to_depth_bwd(Act(s), n, h, w, c).buf
    assert torch.equal(back[..., :c], xb[..., :c])


@pytest.mark.parametrize("shape", [(2, 64, 16, 12), (1, 24, 9, 7), (2, 8, 2, 2)])
def test_maxpool2_fwd_bwd(shape):
    n, c, h, w = shape
    x = bf16r(synth.normalish(shape, 5, "x")).requires_grad_(True)
    ref = F.max_pool2d(x, 2)
    g = bf16r(synth.normalish(tuple(ref.shape), 5, "g"))
    ref.backward(g)
    xb = _to_buf(x.detach())
    y = ops.maxpool2(Act(xb))
    assert torch.equal(y.buf[..., :c].float().cpu(), ref.detach().permute(0, 2, 3, 1))
    dx = ops.maxpool2_bwd(Act(xb), Act(_to_buf(g)))
    assert torch.equal(dx.buf[..., :c].float().cpu(), x.grad.permute(0, 2, 3, 1))


@pytest.mark.parametrize("shape", [(2, 10, 16, 12), (1, 19, 9, 7), (1, 8, 2, 3)])
def test_avgpool3s2_bwd(shape):
    n, c, h, w = shape
    x = bf16r(synth.normalish(shape, 6, "x")).requires_grad_(True)
    ref = F.avg_pool2d(x, 3, stride=2, padding=1, count_include_pad=False)
    g = bf16r(synth.normalish(tuple(ref.shape), 6, "g"))
    ref.backward(g)
    dx = ops.avgpool3s2_bwd(Act(_to_buf(g)), h, w)
    got = dx.buf[..., :c].float().cpu()
    want = x.grad.permute(0, 2, 3, 1)
    assert float((got - want).abs().max()) <= 2 ** -8 * float(want.abs().max()) + 1e-6  # one bf16 rounding of the result


def test_parse_blur_argmax_matches_the_torch_pipeline():
    """train_generator.py:247-273: resize -> Gaussian -> argmax -> one-hot regroup.  The fused kernel must pick the same class
    as the unfused fp32 pipeline except where the two top scores are within float rounding of each other."""
    from hrviton_b200 import train_step
    n, H, W = 2, 160, 96
    seg = synth.normalish((n, 13, 40, 24), 7, "seg").to(DEV)
    idx, onehot = ops.parse_blur_argmax(seg, (H, W), group_of=train_step.GROUP_OF_13, groups=7)
    up = F.interpolate(seg, size=(H, W), mode="bilinear")
    gauss = train_step.gaussian_blur_15_3(up)
    ref = gauss.argmax(1, keepdim=True)
    diff = idx != ref
    if bool(diff.any()):  # disagreements only at numerical ties of the two best classes
        top2 = gauss.topk(2, dim=1).values
        gap = (top2[:, 0] - top2[:, 1])[diff[:, 0]]
        assert float(gap.max()) < 1e-5, float(gap.max())
    assert float(diff.float().mean()) < 1e-3
    # one-hot output == regrouped one-hot of the kernel's own arg-max (exact)
    m = torch.zeros(7, 13, device=DEV)
    for i, grp in enumerate(train_step.LABELS7):
        m[i, grp] = 1.0
    old = torch.zeros(n, 13, H, W, device=DEV).scatter_(1, idx, 1.0)
    assert torch.equal(onehot, torch.einsum("ij,njhw->nihw", m, old))
    # a non multiple-of-tile extent
    idx2, _ = ops.parse_blur_argmax(seg, (50, 45))
    ref2 = train_step.gaussian_blur_15_3(F.interpolate(seg, size=(50, 45), mode="bilinear")).argmax(1, keepdim=True)
    assert float((idx2 != ref2).float().mean()) < 2e-3


@pytest.mark.parametrize("dgrad", [False, True])
@pytest.mark.parametrize("inter", [False, True])
def test_pack_conv_weight(dgrad, inter):
    cout, cin, k = 20, 13, 3
    w0 = synth.normalish((cout, cin, k, k), 8, "w0").to(DEV)
    w1 = synth.normalish((cout, cin, k, k), 8, "w1").to(DEV) if inter else None
    pw = ops.pack_weight(w0, (1, 1), interleave=w1, dgrad=dgrad)
    full = torch.stack([w0, w1], 1).reshape(2 * cout, cin, k, k) if inter else w0  # interleaved rows
    if dgrad:
        full = full.flip(2, 3).transpose(0, 1)  # (cin, cout*, kh, kw)
    rows, cols = full.shape[:2]
    want = torch.zeros_like(pw.w, dtype=torch.float32)
    want[:, :rows, :cols] = full.permute(2, 3, 0, 1).reshape(k * k, rows, cols)
    assert pw.n_gemm == rows
    assert torch.equal(pw.w.float(), want.to(torch.bfloat16).float())


@pytest.mark.parametrize("shape", [(2, 7, 12, 9), (1, 3, 8, 8)])
def test_im2col_conv_equals_direct_conv(shape):
    """hrv_im2col + 1x1 GEMM == the 3x3 convolution it replaces (same products, fp32 accumulation)."""
    n, c, h, w = shape
    x = bf16r(synth.normalish(shape, 9, "x"))
    wt = bf16r(synth.normalish((24, c, 3, 3), 9, "w", 0.2))
    cols = ops.im2col(Act(_to_buf(x), c=c), 3, 3, 1)
    # explicit column check against unfold (channel-major in torch -> tap-major here)
    unf = F.unfold(x, 3, padding=1).reshape(n, c, 9, h, w).permute(0, 3, 4, 2, 1).reshape(n, h, w, 9 * c)
    assert torch.equal(cols.buf[..., :9 * c].float().cpu(), unf)
    assert float(cols.buf[..., 9 * c:].float().abs().max()) == 0.0
    wc = ops.im2col_weight(wt.to(DEV), cols.c)
    out = Act.empty(n, h, w, 24)
    ops.conv2d(cols, ops.pack_weight(wc, (0, 0)), out)
    ref = F.conv2d(x, wt, padding=1)
    assert rel_err(out.to_nchw(), ref) < 1e-2


def test_l1_sum_and_bwd():
    shape = (2, 24, 9, 7)
    a = bf16r(synth.normalish(shape, 10, "a")).requires_grad_(True)
    b = bf16r(synth.normalish(shape, 10, "b"))
    ref = (a - b).abs().mean()
    ref.backward()
    A, B = Act(_to_buf(a.detach())), Act(_to_buf(b))
    s = ops.l1_sum(A, B)
    assert abs(float(s) / a.numel() - float(ref)) < 1e-6
    gs = torch.full((1,), 0.5 / a.numel(), device=DEV)
    da = ops.l1_bwd(A, B, gs).buf.float().cpu().permute(0, 3, 1, 2)
    want = (a.grad * 0.5).to(torch.bfloat16).float()
    assert torch.equal(da, want)


PIXN_CASES = [  # n, cin, cout, h, w, k, pad, act, bias, scale, out_pitch
    (2, 80, 32, 40, 24, 3, 1, 2, True, False, None),     # SW128 K padding 80 -> 128, partial tiles
    (1, 48, 32, 64, 48, 3, 1, 0, True, True, None),
    (3, 160, 128, 17, 13, 3, 1, 1, True, False, None),   # odd extents, odd number of 128-pixel boxes
    (8, 64, 128, 8, 6, 1, 0, 1, True, False, None),      # several images per box (tiny pyramid level)
    (2, 64, 3, 32, 24, 3, 1, 3, True, False, None),      # 3 output channels (pad channels written as zero)
    (1, 256, 128, 33, 25, 2, 1, 2, False, False, None),  # the 2x2/pad-1 form of the stride-2 convolutions (extent H+1)
    (2, 40, 72, 20, 20, 4, 2, 0, True, False, None),     # 4x4 / pad 2 (PatchGAN stride-1 layers), cout not a multiple of 16
    (1, 128, 64, 48, 40, 3, 1, 0, False, False, 96),     # output into a wider buffer (channel slice of a concat buffer)
]


@pytest.mark.parametrize("case", PIXN_CASES)
def test_conv_pixn_matches_classic_kernel(case):
    """The pixel-N kernel (weights as the MMA's M operand, 256 pixels as N, transposed epilogue) accumulates the same products in
    the same K order as the classic kernel: outputs must be bit-identical.  HRV_CONV_PIXN=0 selects the classic kernel."""
    n, cin, cout, h, w, k, pad, act, bias, scale, out_pitch = case
    x = Act(_to_buf(bf16r(synth.normalish((n, cin, h, w), 11, "x"))), c=cin)
    wt = synth.normalish((cout, cin, k, k), 11, "w", (1.0 / (cin * k * k)) ** 0.5).to(DEV)
    b = synth.normalish((cout,), 11, "b", 0.1).to(DEV) if bias else None
    sc = synth.uniform((cout,), 11, "s", 0.5, 1.5).to(DEV) if scale else None
    pw = ops.pack_weight(wt, (pad, pad))
    assert pw.bk == 64
    oh, ow = h + 2 * pad - k + 1, w + 2 * pad - k + 1
    outs = []
    try:
        os.environ["HRV_CONV_HALO"] = "0"  # classic kernel in tap-by-tap order: the same fp32 accumulation order as the pixel-N kernel
        for flag in ("0", "1"):
            os.environ["HRV_CONV_PIXN"] = flag
            o = Act(torch.zeros((n, oh, ow, out_pitch or ops.round_up(cout, 8)), dtype=torch.bfloat16, device=DEV), c=cout)
            ops.conv2d(x, pw, o, act=act, scale=sc, shift=b)
            torch.cuda.synchronize()
            outs.append(o.buf.clone())
    finally:
        os.environ.pop("HRV_CONV_PIXN", None)
        os.environ.pop("HRV_CONV_HALO", None)
    bad = outs[0] != outs[1]
    assert not bool(bad.any()), "%d mismatching elements, first at %s" % (int(bad.sum()), bad.nonzero()[:4].tolist())
    ref = F.conv2d(x.buf[..., :cin].permute(0, 3, 1, 2).float().cpu(), bf16r(wt.cpu()), None, padding=pad)
    if sc is not None:
        ref = ref * sc.cpu()[None, :, None, None]
    if b is not None:
        ref = ref + b.cpu()[None, :, None, None]
    ref = {0: lambda t: t, 1: torch.relu, 2: lambda t: F.leaky_relu(t, 0.2), 3: torch.tanh}[act](ref)
    assert rel_err(outs[1][..., :cout].permute(0, 3, 1, 2), ref) < 1e-2


def test_gaussian_blur_matches_depthwise_conv():
    """hrv_gaussian_blur vs the restated tgm.image.GaussianBlur (separable depth-wise conv, zero padding) on odd extents."""
    from hrviton_b200 import train_step
    x = torch.randn(2, 5, 70, 45)
    got = ops.gaussian_blur(x.cuda(), 15, 3.0).cpu()
    want = train_step.gaussian_blur_15_3(x)
    assert float((got - want).abs().max()) < 2e-6
    k = torch.arange(7, dtype=torch.float32) - 3
    g = torch.exp(-(k * k) / (2 * 1.5 * 1.5))
    g = g / g.sum()
    w2 = torch.nn.functional.conv2d(torch.nn.functional.conv2d(x, g.view(1, 1, 1, 7).expand(5, 1, 1, 7), padding=(0, 3), groups=5),
                                    g.view(1, 1, 7, 1).expand(5, 1, 7, 1), padding=(3, 0), groups=5)
    assert float((ops.gaussian_blur(x.cuda(), 7, 1.5).cpu() - w2).abs().max()) < 2e-6


@pytest.mark.parametrize("shape", [((2, 32, 24), (256, 192), 3), ((1, 128, 96), (1024, 768), 4), ((1, 16, 12), (50, 37), 1)])
def test_flow_warp_nchw_matches_torch_chain(shape):
    """hrv_flow_warp_nchw (flow up-sampling at any scale + normalise + base grid + grid_sample, train_generator.py:232-238) against the
    separate torch ops of the reference on the CPU: grid to 2e-6, sampled values to 1e-5 (|src| <= 1)."""
    import torch.nn.functional as F
    (n, hl, wl), (H, W), c = shape
    g = torch.Generator().manual_seed(5)
    flow = (torch.rand((n, hl, wl, 2), generator=g) - 0.5) * 20.0
    src = torch.rand((n, c, H, W), generator=g) * 2 - 1
    div = ((wl - 1.0) / 2.0, (hl - 1.0) / 2.0)
    up = F.interpolate(flow.permute(0, 3, 1, 2), size=(H, W), mode="bilinear").permute(0, 2, 3, 1)
    gx = torch.linspace(-1.0, 1.0, W).view(1, 1, W, 1).expand(n, H, W, 1)
    gy = torch.linspace(-1.0, 1.0, H).view(1, H, 1, 1).expand(n, H, W, 1)
    grid = torch.cat([up[..., 0:1] / div[0], up[..., 1:2] / div[1]], 3) + torch.cat([gx, gy], 3)
    want = F.grid_sample(src, grid, padding_mode="border", align_corners=False)
    got, ggrid = ops.flow_warp_nchw(flow.cuda(), src.cuda(), (H, W), div, want_grid=True)
    assert float((ggrid.cpu() - grid).abs().max()) < 2e-6
    # a sample coordinate within 2e-6 (normalised) of a pixel boundary may floor differently: compare values, which are continuous
    assert float((got.cpu() - want).abs().max()) < 2e-3 and float((got.cpu() - want).abs().mean()) < 1e-5


@pytest.mark.parametrize("shift,c1,norms", [(1, 16, 2), (1, 16, 1), (0, 0, 2), (0, 8, 1), (1, 0, 2)])
def test_instnorm_stats2_matches_fp64_statistics(shift, c1, norms):
    """hrv_instnorm_stats2 (one pass over the SOURCE tensors, up to two norms with their own noise) against fp64 statistics of the
    materialised virtual tensor cat(up2(x0), x1) + noise_j * ns_j (network_generator.py:101-113)."""
    n, H, W, c0 = 2, 36, 20, 24
    g = torch.Generator().manual_seed(3)
    x0 = bf16r(torch.randn((n, c0, H >> shift, W >> shift), generator=g) * 2 + 0.5)
    x1 = bf16r(torch.randn((n, c1, H, W), generator=g)) if c1 else None
    full = F.interpolate(x0, scale_factor=2, mode="nearest") if shift else x0
    if x1 is not None:
        full = torch.cat([full, x1], 1)
    C = c0 + c1
    noises = [torch.randn((n, H, W), generator=g) for _ in range(norms)]
    nss = [torch.randn(C, generator=g) * 0.3 for _ in range(norms)]
    to_act = lambda t: Act(t.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16).to(DEV))
    outs = ops.instnorm_stats2(to_act(x0), shift, to_act(x1) if x1 is not None else None, H, W, [z.to(DEV) for z in noises],
                               [s.to(DEV) for s in nss])
    for j in range(norms):
        v = (full + noises[j][:, None] * nss[j][None, :, None, None]).double()
        m = v.mean((2, 3))
        r = 1.0 / torch.sqrt(v.var((2, 3), unbiased=False) + 1e-5)
        assert float((outs[j][0].cpu().double() - m).abs().max()) < 2e-5
        assert float(((outs[j][1].cpu().double() - r) / r).abs().max()) < 2e-5
    # without noise it reproduces the plain InstanceNorm statistics of the first kernel
    plain = ops.instnorm_stats2(to_act(x0), shift, to_act(x1) if x1 is not None else None, H, W, [None], [None])[0]
    ref = ops.instnorm_stats(to_act(x0), shift, to_act(x1) if x1 is not None else None, H, W, None, None)
    assert float((plain[0] - ref[0]).abs().max()) < 1e-5 and float(((plain[1] - ref[1]) / ref[1]).abs().max()) < 1e-5


def test_onehot_u8():
    lab = torch.randint(0, 13, (3, 1, 37, 29), dtype=torch.uint8)
    got = ops.onehot_u8(lab.to(DEV), 13).cpu()
    want = torch.zeros(3, 13, 37, 29).scatter_(1, lab.long(), 1.0)
    assert torch.equal(got, want)


def test_conv_wgrad_is_bit_reproducible():
    """Split-K partial tiles go to private workspace slabs and are summed in a fixed order (round 1 used fp32 atomics): two runs on the
    same data give bit-identical dW, also for a layer whose element count is not a multiple of 4 (scalar reduction path)."""
    for cin, cout, k, h, w in [(128, 160, 3, 192, 144), (13, 13, 3, 96, 80), (64, 128, 1, 256, 192)]:
        x = Act(torch.randn(2, h, w, ops.round_up(cin, 8), device=DEV).to(torch.bfloat16), c=cin)
        dy = Act(torch.randn(2, h, w, ops.round_up(cout, 8), device=DEV).to(torch.bfloat16), c=cout)
        a = ops.conv2d_wgrad(x, dy, k, k, k // 2).clone()
        for _ in range(3):
            b = ops.conv2d_wgrad(x, dy, k, k, k // 2)
            assert torch.equal(a, b), (cin, cout, k)
        ref = torch.nn.grad.conv2d_weight(x.buf[..., :cin].permute(0, 3, 1, 2).float(), (cout, cin, k, k),
                                          dy.buf[..., :cout].permute(0, 3, 1, 2).float(), padding=k // 2)
        assert rel_err(a, ref) < 2e-3


PAIR_CASES = [  # spade, cin, n_gemm, h, w, batch, x0_shift, c1 (x1 channels)
    (True, 128, 160, 64, 48, 2, 0, 0), (True, 128, 160, 64, 48, 2, 1, 16), (True, 128, 288, 48, 32, 3, 1, 16),
    (True, 128, 544, 64, 48, 2, 1, 16),    # bn 192: two TMEM accumulators, two owner warpgroups
    (True, 128, 2080, 16, 12, 2, 1, 16),   # 13 N tiles, more channels than the shared-memory constant table holds (global-load path)
    (True, 128, 144, 30, 22, 1, 0, 0),     # odd number of pixel tiles: the pair's second CTA runs a tile past the end
    (False, 160, 160, 50, 37, 3, 0, 0), (False, 256, 256, 64, 48, 2, 0, 0), (False, 80, 192, 128, 96, 1, 0, 0),
    # narrow tiles (32 / 64 / 128 columns: 16 / 32 / 64 weight rows per CTA)
    (True, 128, 64, 64, 48, 2, 1, 16), (True, 128, 128, 48, 32, 2, 0, 0), (False, 80, 32, 64, 48, 2, 0, 0), (False, 144, 64, 50, 37, 2, 0, 0),
    (False, 160, 128, 64, 48, 1, 0, 0), (False, 2080, 128, 16, 12, 2, 0, 0)]


@pytest.mark.parametrize("case", PAIR_CASES)
def test_conv_pair_kernel_matches_single_cta_kernel(case):
    """The CTA-pair kernel (tcgen05 cta_group::2: M = 256 over two SMs, each CTA holding half of every weight stage; epilogue
    warpgroup w drains accumulator w) against the one-CTA kernel on identical inputs (HRV_CONV_PAIR=0).  Same products, and — when the
    one-CTA kernel also runs its halo mainloop (tiles of <= 32 or 144..208 columns) — the same fp32 accumulation order: bit-identical
    outputs, gamma included.  Elsewhere the one-CTA kernel walks K tap by tap: equal to one bf16 ulp."""
    spade, cin, ng, h, w, B, shift, c1 = case
    g = torch.Generator().manual_seed(1)
    rnd = lambda *s: torch.randn(*s, generator=g)
    x = Act(rnd(B, h, w, ops.round_up(cin, 8)).to(torch.bfloat16).to(DEV), c=cin)
    outs = []
    try:
        os.environ["HRV_CONV_PIXN"] = "0"
        if spade:
            C = ng // 2
            pw = ops.pack_weight((rnd(C, cin, 3, 3) * 0.05).to(DEV), (1, 1), interleave=(rnd(C, cin, 3, 3) * 0.05).to(DEV))
            x0 = Act(rnd(B, h >> shift, w >> shift, C - c1).to(torch.bfloat16).to(DEV))
            x1 = Act(rnd(B, h, w, c1).to(torch.bfloat16).to(DEV)) if c1 else None
            mean, rstd = (rnd(B, C) * 0.1).to(DEV), (torch.rand(B, C, generator=g) + 0.5).to(DEV)
            noise, ns, sh = rnd(B, h, w).to(DEV), (rnd(C) * 0.1).to(DEV), (rnd(2 * C) * 0.1).to(DEV)
        else:
            pw = ops.pack_weight((rnd(ng, cin, 3, 3) * 0.05).to(DEV), (1, 1))
            bias = rnd(ng).to(DEV)
        if pw.bk != 64:
            pytest.skip("the pair kernel needs 64-channel K blocks")
        for flag in ("0", "1"):
            os.environ["HRV_CONV_PAIR"] = flag
            if spade:
                out, gam = Act.empty(B, h, w, C, zero=True), Act.empty(B, h, w, C, zero=True)
                ops.conv2d_spade(x, pw, out, x0, shift, x1, mean, rstd, noise, ns, sh, 2, gamma_out=gam)
                torch.cuda.synchronize()
                outs.append((out.buf.float().clone(), gam.buf.float().clone()))
            else:
                out = Act.empty(B, h, w, ng, zero=True)
                ops.conv2d(x, pw, out, act=2, shift=bias)
                torch.cuda.synchronize()
                outs.append((out.buf.float().clone(), None))
    finally:
        os.environ.pop("HRV_CONV_PAIR", None)
        os.environ.pop("HRV_CONV_PIXN", None)
    (a, ga), (b, gb) = outs
    d = float((a - b).abs().max())
    if pw.bn <= 32 or 144 <= pw.bn <= 208:  # the one-CTA kernel runs the halo mainloop too: same accumulation order
        assert d == 0.0 and (ga is None or float((ga - gb).abs().max()) == 0.0)
    else:  # tap-by-tap K order in the one-CTA kernel: fp32 sums differ in the last bits -> at most one bf16 ulp of the largest output
        assert d <= 2 ** -7 * float(a.abs().max())
        assert ga is None or float((ga - gb).abs().max()) <= 2 ** -7 * float(ga.abs().max())


def test_feature_matching_term_matches_torch():
    """autograd_g.FeatMatchFn (hrv_l1_sum / hrv_l1_bwd over the [fake; real] halves of one discriminator feature buffer) against the
    reference expression of train_generator.py:303-311, value and gradient (the real half gets exactly zero)."""
    from hrviton_b200 import autograd_g
    g = torch.Generator().manual_seed(5)
    buf = torch.randn(6, 33, 25, 64, generator=g).to(torch.bfloat16).to(DEV).requires_grad_(True)
    loss = autograd_g.FeatMatchFn.apply(buf) * 2.5
    loss.backward()
    ref_in = buf.detach().float().requires_grad_(True)
    v = ref_in.permute(0, 3, 1, 2)
    ref = (v[:3] - v[3:].detach()).abs().mean() * 2.5
    ref.backward()
    assert abs(float(loss) - float(ref)) < 1e-5 * abs(float(ref))
    got, want = buf.grad.float(), ref_in.grad
    assert float(got[3:].abs().max()) == 0.0
    # sign(a-b) * 2.5 / numel, rounded to bf16 once
    assert torch.allclose(got[:3], want[:3].to(torch.bfloat16).float(), rtol=0, atol=0)
