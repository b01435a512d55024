"""NHWC activation views + thin wrappers over the C-ABI.  torch is used here for device memory and streams only."""
import ctypes
from dataclasses import dataclass

import torch
import torch.nn.functional as F

from . import capi
from .capi import ACT_LRELU, ACT_NONE, ACT_RELU, ACT_TANH, BF16, F32  # noqa: F401

LAUNCHES = [0]  # count of kernel launches issued through the C-ABI (bench.py reads this for `gpu_launches`)
PARAM_GEN = [0]  # generation of the parameter values: part of every derived-weight cache key (spade._param_key)
STORAGE = [torch.bfloat16]  # activation storage type of newly created buffers: torch.bfloat16 (default) or torch.float16
PROFILE = None  # bench.py sets this to a list; every C-ABI call then appends (kind, work, start_event, end_event)


class _Timed:
    """Brackets one C-ABI call with CUDA events on the launching stream when profiling is on (bench.py roofline)."""

    def __init__(self, kind, work, launches=1, label=""):
        self.kind, self.work, self.launches, self.label = kind, work, launches, label

    def __enter__(self):
        LAUNCHES[0] += self.launches
        if PROFILE is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *exc):
        if PROFILE is not None:
            self.e1.record()
            PROFILE.append((self.kind, self.work, self.e0, self.e1, self.label))
        return False


def set_precision(name):
    """'bf16' (default: bf16 activations, fp32 accumulation — the training configuration) or 'fp16' (IEEE half activations,
    3 more mantissa bits: the storage type of the reference's own apex-O1 --fp16 runs, train_generator.py:161-169; meets the
    1e-2 forward tolerance of BASELINE.json).  Invalidates every derived-weight cache."""
    dt = {"bf16": torch.bfloat16, "fp16": torch.float16}[name]
    if STORAGE[0] != dt:
        STORAGE[0] = dt
        PARAM_GEN[0] += 1


def get_precision():
    return "fp16" if STORAGE[0] == torch.float16 else "bf16"


def _L(*things):
    """The library flavour matching the storage type of the given Acts / tensors (fp16 if any of them is torch.float16)."""
    for t in things:
        if t is None:
            continue
        d = t.buf.dtype if isinstance(t, Act) else (t.dtype if torch.is_tensor(t) else t)
        if d == torch.float16:
            return capi.lib(torch.float16)
    return capi.lib()


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def round_up(v, m):
    return (v + m - 1) // m * m


class Act:
    """A pixel-major (NHWC) activation: `buf` is (N,H,W,P) bf16|fp32 on the GPU; the view covers channels
    [c0, c0+c) of every pixel.  Channel slices of one buffer replace torch.cat."""

    def __init__(self, buf, c=None, c0=0):
        assert buf.is_cuda and buf.dim() == 4 and buf.is_contiguous(), "Act needs a contiguous CUDA (N,H,W,P) buffer"
        self.buf = buf
        self.c0 = c0
        self.c = buf.shape[3] - c0 if c is None else c
        assert self.c0 + self.c <= buf.shape[3]

    @staticmethod
    def empty(n, h, w, c, dtype=None, device="cuda", pitch=None, zero=False):
        dtype = STORAGE[0] if dtype is None else dtype
        p = round_up(c, 8) if pitch is None else pitch
        f = torch.zeros if zero else torch.empty
        return Act(f((n, h, w, p), dtype=dtype, device=device), c=c)

    n = property(lambda s: s.buf.shape[0])
    h = property(lambda s: s.buf.shape[1])
    w = property(lambda s: s.buf.shape[2])
    pitch = property(lambda s: s.buf.shape[3])

    def slice(self, c0, c):
        return Act(self.buf, c=c, c0=self.c0 + c0)

    def ct(self):
        es = self.buf.element_size()
        return capi.Tensor(self.buf.data_ptr() + self.c0 * es, self.n, self.h, self.w, self.c, self.pitch,
                           F32 if self.buf.dtype == torch.float32 else BF16)

    def to_nchw(self):
        """fp32 NCHW copy (API boundary / tests)."""
        out = torch.empty((self.n, self.c, self.h, self.w), dtype=torch.float32, device=self.buf.device)
        t = self.ct()
        with _Timed("glue", 0.0, label="nhwc_to_nchw"):
            capi.check(_L(self).hrv_nhwc_to_nchw(ctypes.byref(t), out.data_ptr(), _stream()), "nhwc_to_nchw")
        return out


_NULL = capi.Tensor(None, 0, 0, 0, 0, 0, 0)


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def from_nchw(x, c_pad=None, size=None, out=None):
    """fp32 NCHW (cuda) -> bf16 NHWC Act, optional nearest resize to `size` (F.interpolate nearest)."""
    assert x.is_cuda and x.dtype == torch.float32
    x = x.contiguous()
    n, c, h, w = x.shape
    oh, ow = (h, w) if size is None else size
    if out is None:
        out = Act.empty(n, oh, ow, c, pitch=round_up(c if c_pad is None else c_pad, 8))
    t = out.ct()
    with _Timed("glue", 0.0, label="nchw_to_nhwc"):
        capi.check(_L(out).hrv_nchw_to_nhwc(x.data_ptr(), c, h, w, ctypes.byref(t), _stream()), "nchw_to_nhwc")
    return out


# ----------------------------------------------------------------------------------------------- weights

def pick_bk(cin):
    cands = [64, 32] + ([16] if cin <= 16 else [])
    pads = {bk: round_up(cin, bk) for bk in cands}
    best = min(pads.values())
    for bk in cands:
        if pads[bk] <= 1.10 * best:
            return bk
    return cands[-1]


def pick_bn(n_gemm):
    n16 = round_up(n_gemm, 16)
    if n16 <= 256:
        return n16
    # cost model: every N tile re-streams the A operand once (+64 ~ fixed per-tile overhead in columns)
    best, best_cost = 256, None
    for bn in range(256, 15, -16):
        tiles = (n_gemm + bn - 1) // bn
        cost = (tiles * (bn + 64), tiles * bn)
        if best_cost is None or cost < best_cost:
            best, best_cost = bn, cost
    return best


def pick_bn_spade(n_gemm):
    """N tile of a gamma|beta GEMM (n_gemm = 2C interleaved columns).  With several N tiles the staged epilogue of the CTA-pair kernel
    needs each tile's channel range to end on a 16-channel slab, i.e. bn % 32 == 0: take the candidate with the fewest padded columns
    (ties: the wider tile)."""
    n16 = round_up(n_gemm, 16)
    if n16 <= 256:
        return n16
    best = None
    for bn in (256, 224, 192, 160):
        cols = round_up(n_gemm, bn)
        if best is None or cols < best[0]:
            best = (cols, bn)
    return best[1]


@dataclass
class PackedConv:
    w: torch.Tensor  # bf16 [taps, n_pad, cin_k]
    kh: int
    kw: int
    off_y: int
    off_x: int
    bk: int
    bn: int
    n_gemm: int
    cin: int
    flops_per_pixel: float = 0.0  # algorithmic 2*Cin*Cout*kh*kw of the ORIGINAL convolution (unpadded, pre-s2d)


def pack_weight(w, off, cin_total=None, interleave=None, bn=None, flops_per_pixel=None, dgrad=False):
    """w: (Cout,Cin,kh,kw) fp32 cuda (already divided by sigma / transformed). Returns PackedConv (one kernel: hrv_pack_conv_weight).
    interleave: a second weight of identical shape whose rows are interleaved (gamma_c, beta_c pairs).
    dgrad=True packs the operand of the data-gradient convolution (flip + transpose) without materialising it."""
    w = w.detach()
    if w.dtype != torch.float32 or not w.is_contiguous():
        w = w.float().contiguous()
    if interleave is not None:
        interleave = interleave.detach()
        if interleave.dtype != torch.float32 or not interleave.is_contiguous():
            interleave = interleave.float().contiguous()
        assert interleave.shape == w.shape
    cout, cin, kh, kw = w.shape
    inter = 2 if interleave is not None else 1
    rows, cols = (cin, cout * inter) if dgrad else (cout * inter, cin)  # GEMM N rows, K columns
    k_eff = cols if cin_total is None else cin_total
    # Cout <= 128: eligible for the pixel-N kernel (conv_pixn_kernel), which needs 64-channel K blocks (zero padded)
    bk = 64 if (rows <= 128 and k_eff > 32) else pick_bk(k_eff)  # K <= 32 stays on the 32-wide blocks (padding to 64 would double the MMAs)
    cin_k = round_up(k_eff, bk)
    if bn is None:
        bn = pick_bn_spade(rows) if (interleave is not None and not dgrad) else pick_bn(rows)
    n_pad = round_up(rows, bn)
    wp = torch.empty((kh * kw, n_pad, cin_k), dtype=STORAGE[0], device=w.device)
    with _Timed("glue", 0.0, label="pack_conv_weight"):
        capi.check(_L(wp).hrv_pack_conv_weight(w.data_ptr(), _p(interleave), cout, cin, kh, kw, 1 if dgrad else 0, None, wp.data_ptr(),
                                                   n_pad, cin_k, _stream()), "pack_conv_weight")
    fpp = 2.0 * cin * cout * inter * kh * kw if flops_per_pixel is None else flops_per_pixel
    return PackedConv(wp, kh, kw, off[0], off[1], bk, bn, rows, k_eff, fpp)


def s2d_weight(w, pad):
    """Rewrite a stride-2 conv weight (Cout,Cin,k,k) with padding `pad` (k=4,pad=2 or k=3,pad=1) as the
    2x2 stride-1 weight over the space-to-depth input with channel order (py*2+px)*Cin8 + ci, off=(1,1).
    An index shuffle, so gradients flow back to w.  The 3x3 form is the 4x4 one with a zero first row/column
    (tap ky of the 3x3 sits at ky+1)."""
    cout, cin, k, _ = w.shape
    assert (k, pad) in ((4, 2), (3, 1))
    cin8 = round_up(cin, 8)
    wp = F.pad(w, (4 - k, 0, 4 - k, 0, 0, cin8 - cin)).reshape(cout, cin8, 2, 2, 2, 2)  # ky = ty*2+py, kx = tx*2+px
    return wp.permute(0, 3, 5, 1, 2, 4).reshape(cout, 4 * cin8, 2, 2)  # channel = (py*2+px)*cin8 + ci, taps (ty,tx)


def im2col_weight(w, k_pad):
    """(cout,cin,kh,kw) -> (cout,k_pad,1,1) in the tap-major column order of hrv_im2col (differentiable index shuffle)."""
    cout, cin, kh, kw = w.shape
    return F.pad(w.permute(0, 2, 3, 1).reshape(cout, kh * kw * cin), (0, k_pad - kh * kw * cin)).reshape(cout, k_pad, 1, 1)


def pack_s2d(w, pad):
    """PackedConv of a stride-2 convolution expressed on the space-to-depth input (algorithmic FLOPs of the original)."""
    cout, cin, k, _ = w.shape
    return pack_weight(s2d_weight(w, pad), (1, 1), flops_per_pixel=2.0 * cin * cout * k * k)


# ----------------------------------------------------------------------------------------------- ops

def conv2d(inp, pw, out, act=ACT_NONE, scale=None, shift=None, res=None, out_layout=capi.NHWC, res_mode=capi.RES_ADD):
    assert inp.c == pw.cin, (inp.c, pw.cin)
    p = capi.ConvParams()
    p.inp = inp.ct()
    p.wpack = pw.w.data_ptr()
    p.kh, p.kw, p.off_y, p.off_x = pw.kh, pw.kw, pw.off_y, pw.off_x
    p.bk, p.bn, p.n_gemm = pw.bk, pw.bn, pw.n_gemm
    if isinstance(out, Act):
        p.out = out.ct()
    else:  # raw fp32 NCHW torch tensor
        n, c, h, w = out.shape
        p.out = capi.Tensor(out.data_ptr(), n, h, w, c, c, F32)
    p.out_layout = out_layout
    p.epi = capi.EPI_LINEAR
    p.act = act
    p.scale = _p(scale)
    p.shift = _p(shift)
    p.res = res.ct() if res is not None else _NULL
    p.res_mode = res_mode if res is not None else 0
    p.x0 = _NULL
    p.x1 = _NULL
    p.gamma_out = _NULL
    with _Timed("conv", pw.flops_per_pixel * p.out.n * p.out.h * p.out.w,
                label="%d->%d k%dx%d n%d %dx%d bk%d bn%d" % (inp.c, pw.n_gemm, pw.kh, pw.kw, p.out.n, p.out.h, p.out.w, pw.bk, pw.bn)):
        capi.check(_L(inp).hrv_conv2d_fwd(ctypes.byref(p), _stream()), "conv2d_fwd")
    return out


def conv2d_spade(actv, pw, out, x0, x0_shift, x1, mean, rstd, noise, noise_scale, shift, act, gamma_out=None):
    p = capi.ConvParams()
    p.inp = actv.ct()
    p.wpack = pw.w.data_ptr()
    p.kh, p.kw, p.off_y, p.off_x = pw.kh, pw.kw, pw.off_y, pw.off_x
    p.bk, p.bn, p.n_gemm = pw.bk, pw.bn, pw.n_gemm
    p.out = out.ct()
    p.out_layout = capi.NHWC
    p.epi = capi.EPI_SPADE
    p.act = act
    p.scale = None
    p.shift = _p(shift)
    p.res = _NULL
    p.res_mode = 0
    p.x0 = x0.ct()
    p.x1 = x1.ct() if x1 is not None else _NULL
    p.x0_shift = x0_shift
    p.mean, p.rstd, p.noise, p.noise_scale = _p(mean), _p(rstd), _p(noise), _p(noise_scale)
    p.gamma_out = gamma_out.ct() if gamma_out is not None else _NULL
    with _Timed("conv_spade", pw.flops_per_pixel * out.n * out.h * out.w,
                label="%d->%d k%dx%d n%d %dx%d bk%d bn%d" % (actv.c, pw.n_gemm, pw.kh, pw.kw, out.n, out.h, out.w, pw.bk, pw.bn)):
        capi.check(_L(actv).hrv_conv2d_fwd(ctypes.byref(p), _stream()), "conv2d_fwd(spade)")
    return out


_ws = {}


def _workspace(nbytes, device):
    key = (device, "ws")
    w = _ws.get(key)
    if w is None or w.numel() < nbytes:
        w = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
        _ws[key] = w
    return w


def instnorm_stats(x0, x0_shift, x1, h, w, noise, noise_scale, eps=1e-5):
    n = x0.n
    c = x0.c + (x1.c if x1 is not None else 0)
    mean = torch.empty((n, c), dtype=torch.float32, device=x0.buf.device)
    rstd = torch.empty_like(mean)
    ws = _workspace(n * c * 16, x0.buf.device)
    t0 = x0.ct()
    t1 = x1.ct() if x1 is not None else _NULL
    nbytes = n * h * w * (2.0 * c + (4.0 if noise is not None else 0.0))  # one bf16 read of every element (+ noise)
    with _Timed("instnorm_stats", nbytes, launches=3, label="c%d n%d %dx%d shift%d" % (c, n, h, w, x0_shift)):
        capi.check(_L(x0).hrv_instnorm_stats(ctypes.byref(t0), x0_shift, ctypes.byref(t1), h, w, _p(noise), _p(noise_scale),
                                                 eps, mean.data_ptr(), rstd.data_ptr(), ws.data_ptr(), ws.numel(), _stream()),
                   "instnorm_stats")
    return mean, rstd


def instnorm_stats2(x0, x0_shift, x1, h, w, noises, noise_scales, eps=1e-5):
    """Statistics of one or two SPADE norms sharing the input cat(up2^shift(x0), x1) (hrv_instnorm_stats2): `noises` / `noise_scales`
    are lists of 1 or 2 entries (a noise entry may be None).  Returns [(mean, rstd), ...] in the same order."""
    n = x0.n
    c = x0.c + (x1.c if x1 is not None else 0)
    k = len(noises)
    assert k in (1, 2) and len(noise_scales) == k
    dev = x0.buf.device
    outs = [(torch.empty((n, c), dtype=torch.float32, device=dev), torch.empty((n, c), dtype=torch.float32, device=dev)) for _ in range(k)]
    ws = _workspace((n * c * 4 + n * 4) * 8, dev)
    t0 = x0.ct()
    t1 = x1.ct() if x1 is not None else _NULL
    src_bytes = 2.0 * n * (x0.h * x0.w * x0.c + (h * w * x1.c if x1 is not None else 0)) + 4.0 * n * h * w * sum(z is not None for z in noises)
    nz1, ns1, m1, r1 = (noises[1], noise_scales[1], outs[1][0], outs[1][1]) if k == 2 else (None, None, None, None)
    with _Timed("instnorm_stats", src_bytes, launches=3 + (1 if x1 is not None else 0), label="c%d n%d %dx%d shift%d norms%d" % (c, n, h, w, x0_shift, k)):
        capi.check(_L(x0).hrv_instnorm_stats2(ctypes.byref(t0), x0_shift, ctypes.byref(t1), h, w, _p(noises[0]), _p(noise_scales[0]), _p(nz1), _p(ns1),
                                              eps, outs[0][0].data_ptr(), outs[0][1].data_ptr(), _p(m1), _p(r1), ws.data_ptr(), ws.numel(), _stream()),
                   "instnorm_stats2")
    return outs


def instnorm_apply(x, mean, rstd, act, out=None):
    out = x if out is None else out
    tx, ty = x.ct(), out.ct()
    with _Timed("glue", 0.0, label="instnorm_apply"):
        capi.check(_L(x).hrv_instnorm_apply(ctypes.byref(tx), mean.data_ptr(), rstd.data_ptr(), act, ctypes.byref(ty), _stream()),
                   "instnorm_apply")
    return out


def space_to_depth(x):
    out = Act.empty(x.n, (x.h + 1) // 2, (x.w + 1) // 2, 4 * round_up(x.c, 8))
    tx, ty = x.ct(), out.ct()
    with _Timed("glue", 0.0, label="space_to_depth"):
        capi.check(_L(x).hrv_space_to_depth(ctypes.byref(tx), ctypes.byref(ty), _stream()), "space_to_depth")
    return out


def space_to_depth_bwd(d, n, h, w, c, pitch=None):
    """dx (n,h,w,c) of space_to_depth from the gradient d of its (n,ceil(h/2),ceil(w/2),4*c8) output."""
    dx = Act.empty(n, h, w, c, pitch=pitch)
    td, tx = d.ct(), dx.ct()
    with _Timed("glue", 0.0, label="space_to_depth_bwd"):
        capi.check(_L(d).hrv_space_to_depth_bwd(ctypes.byref(td), ctypes.byref(tx), _stream()), "space_to_depth_bwd")
    return dx


def maxpool2(x):
    y = Act.empty(x.n, x.h // 2, x.w // 2, x.c, pitch=x.pitch if x.c0 == 0 else None)
    tx, ty = x.ct(), y.ct()
    with _Timed("glue", 0.0, label="maxpool2_fwd"):
        capi.check(_L(x).hrv_maxpool2_fwd(ctypes.byref(tx), ctypes.byref(ty), _stream()), "maxpool2_fwd")
    return y


def maxpool2_bwd(x, dy, relu_gate=False):
    dx = Act.empty(x.n, x.h, x.w, x.c, pitch=x.pitch if x.c0 == 0 else None)
    tx, tdy, tdx = x.ct(), dy.ct(), dx.ct()
    with _Timed("glue", 0.0, label="maxpool2_bwd"):
        capi.check(_L(x).hrv_maxpool2_bwd(ctypes.byref(tx), ctypes.byref(tdy), ctypes.byref(tdx), 1 if relu_gate else 0, _stream()), "maxpool2_bwd")
    return dx


def avgpool3s2_bwd(dy, h, w):
    dx = Act.empty(dy.n, h, w, dy.c, pitch=dy.pitch if dy.c0 == 0 else None)
    tdy, tdx = dy.ct(), dx.ct()
    with _Timed("glue", 0.0, label="avgpool3s2_bwd"):
        capi.check(_L(dy).hrv_avgpool3s2_bwd(ctypes.byref(tdy), ctypes.byref(tdx), _stream()), "avgpool3s2_bwd")
    return dx


def im2col(x, kh, kw, pad, k_pad=None):
    """(n,h,w,c) -> (n,h,w,K) with K = round_up(kh*kw*c, 64|32|16): the tap-major column form of a tiny-Cin convolution."""
    k = kh * kw * x.c
    if k_pad is None:
        k_pad = round_up(k, 64) if k > 32 else (32 if k > 16 else 16)
    out = Act.empty(x.n, x.h, x.w, k_pad)
    tx, to = x.ct(), out.ct()
    with _Timed("glue", 0.0, label="im2col"):
        capi.check(_L(x).hrv_im2col(ctypes.byref(tx), ctypes.byref(to), kh, kw, pad, _stream()), "im2col")
    return out


def l1_sum(a, b):
    """sum |a - b| as a 1-element fp64 cuda tensor."""
    out = torch.empty(1, dtype=torch.float64, device=a.buf.device)
    ta, tb = a.ct(), b.ct()
    with _Timed("glue", 0.0, label="l1_sum"):
        capi.check(_L(a).hrv_l1_sum(ctypes.byref(ta), ctypes.byref(tb), out.data_ptr(), _stream()), "l1_sum")
    return out


def l1_bwd(a, b, gscale, relu_gate=False, out=None):
    """da = sign(a - b) * gscale (gscale: 1-element fp32 cuda tensor); relu_gate: times (a > 0).  out: Act to write into."""
    da = out if out is not None else Act.empty(a.n, a.h, a.w, a.c, pitch=a.pitch if a.c0 == 0 else None)
    ta, tb, td = a.ct(), b.ct(), da.ct()
    with _Timed("glue", 0.0, label="l1_bwd"):
        capi.check(_L(a).hrv_l1_bwd(ctypes.byref(ta), ctypes.byref(tb), gscale.data_ptr(), ctypes.byref(td), 1 if relu_gate else 0, _stream()), "l1_bwd")
    return da


def parse_blur_argmax(seg, size, group_of=None, groups=0, want_idx=True, overlap_classes=None):
    """seg (n,c,h,w) fp32 cuda -> (idx (n,1,H,W) int64 | None, onehot (n,groups,H,W) fp32 | None[, overlap (n,1,H,W)]);
    hrv_parse_blur_argmax.  overlap_classes: class ids whose softmax (over the blurred scores) is summed into `overlap`."""
    assert seg.is_cuda and seg.dtype == torch.float32
    seg = seg.contiguous()
    n, c, h, w = seg.shape
    H, W = size
    idx = torch.empty((n, 1, H, W), dtype=torch.int64, device=seg.device) if want_idx else None
    onehot = torch.empty((n, groups, H, W), dtype=torch.float32, device=seg.device) if group_of is not None else None
    garr = (ctypes.c_int32 * c)(*group_of) if group_of is not None else None
    overlap = torch.empty((n, 1, H, W), dtype=torch.float32, device=seg.device) if overlap_classes else None
    mask = 0
    for k in (overlap_classes or ()):
        mask |= 1 << int(k)
    with _Timed("glue", 0.0, label="parse_blur_argmax"):
        capi.check(capi.lib().hrv_parse_blur_argmax(seg.data_ptr(), n, c, h, w, H, W, garr, groups, _p(idx), _p(onehot), mask, _p(overlap), _stream()),
                   "parse_blur_argmax")
    return (idx, onehot, overlap) if overlap_classes else (idx, onehot)


def onehot_u8(labels, classes, out=None):
    """(N,1,H,W) or (N,H,W) uint8 label map (cuda) -> (N,classes,H,W) fp32 one-hot planes (hrv_onehot_u8): the device half of the
    input feeding — the host ships one byte per pixel instead of `classes` floats (cp_dataset.py:150-172)."""
    assert labels.is_cuda and labels.dtype == torch.uint8
    labels = labels.contiguous()
    n, h, w = labels.shape[0], labels.shape[-2], labels.shape[-1]
    if out is None:
        out = torch.empty((n, classes, h, w), dtype=torch.float32, device=labels.device)
    assert out.is_contiguous() and out.shape == (n, classes, h, w)
    with _Timed("glue", 0.0, label="onehot_u8"):
        capi.check(capi.lib().hrv_onehot_u8(labels.data_ptr(), n, classes, h, w, out.data_ptr(), _stream()), "onehot_u8")
    return out


def gaussian_blur(x, ksize=15, sigma=3.0):
    """tgm.image.GaussianBlur((ksize,ksize),(sigma,sigma)) on an fp32 NCHW cuda tensor (hrv_gaussian_blur)."""
    assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 4
    x = x.contiguous()
    out = torch.empty_like(x)
    n, c, h, w = x.shape
    with _Timed("glue", 0.0, label="gaussian_blur"):
        capi.check(capi.lib().hrv_gaussian_blur(x.data_ptr(), n * c, h, w, ksize, float(sigma), out.data_ptr(), _stream()), "gaussian_blur")
    return out


def flow_warp_nchw(flow_lo, src, size, div_xy, want_grid=False, mask=None, overlap=None, composite=False):
    """The hi-res cloth warp of the glue (train_generator.py:232-238): flow_lo fp32 (N,hl,wl,2) is up-sampled bilinearly to `size`,
    divided by div_xy, added to the linspace base grid and used to grid_sample (bilinear, border) src fp32 (N,C,Hs,Ws).
    mask (N,1,Hs,Ws): the cloth mask is warped with the same taps (returned third), `overlap` (N,1,H,W) applies remove_overlap to it and
    composite=True blends the cloth over white with it (train_generator.py:239-244).
    Returns (warped (N,C,H,W) fp32, grid (N,H,W,2) | None[, warped mask (N,1,H,W)])."""
    assert flow_lo.is_cuda and src.is_cuda and flow_lo.dtype == torch.float32 and src.dtype == torch.float32
    flow_lo, src = flow_lo.contiguous(), src.contiguous()
    n, hl, wl, _ = flow_lo.shape
    _, c, hs, ws = src.shape
    H, W = size
    dev = src.device
    out = torch.empty((n, c, H, W), dtype=torch.float32, device=dev)
    grid = torch.empty((n, H, W, 2), dtype=torch.float32, device=dev) if want_grid else None
    mask_out = None
    if mask is not None:
        mask = mask.float().contiguous()
        assert mask.shape == (n, 1, hs, ws)
        mask_out = torch.empty((n, 1, H, W), dtype=torch.float32, device=dev)
    if overlap is not None:
        overlap = overlap.contiguous()
        assert overlap.shape == (n, 1, H, W) and overlap.dtype == torch.float32
    with _Timed("glue", 0.0, label="flow_warp_nchw"):
        capi.check(capi.lib().hrv_flow_warp_nchw(flow_lo.data_ptr(), n, hl, wl, linspace_table(W, dev).data_ptr(), linspace_table(H, dev).data_ptr(),
                                                 src.data_ptr(), c, hs, ws, out.data_ptr(), H, W, float(div_xy[0]), float(div_xy[1]), _p(grid),
                                                 _p(mask), _p(overlap), _p(mask_out), 1 if composite else 0, _stream()), "flow_warp_nchw")
    return (out, grid, mask_out) if mask is not None else (out, grid)


def avgpool3s2(x):
    out = Act.empty(x.n, (x.h - 1) // 2 + 1, (x.w - 1) // 2 + 1, x.c, pitch=x.pitch if x.c0 == 0 else None)
    tx, ty = x.ct(), out.ct()
    with _Timed("glue", 0.0, label="avgpool3s2"):
        capi.check(_L(x).hrv_avgpool3s2(ctypes.byref(tx), ctypes.byref(ty), _stream()), "avgpool3s2")
    return out


def bilinear_up2_add(a, b, out):
    ta, to = a.ct(), out.ct()
    tb = b.ct() if b is not None else _NULL
    with _Timed("glue", 0.0, label="bilinear_up2_add"):
        capi.check(_L(a).hrv_bilinear_up2_add(ctypes.byref(ta), ctypes.byref(tb), ctypes.byref(to), _stream()), "bilinear_up2_add")
    return out


_lin = {}


def linspace_table(n, device):
    """torch.linspace(-1, 1, n) — the reference's base-grid values (networks.py:162-163), built on the CPU exactly as
    the reference does, cached on the device."""
    key = (n, str(device))
    if key not in _lin:
        _lin[key] = torch.linspace(-1.0, 1.0, n).to(device)
    return _lin[key]


def flow_warp(flow_lo, src, dst, want_flow_up=True, want_idx=False):
    """flow_lo: fp32 (N,h,w,2) cuda contiguous. Returns (flow_up fp32 (N,2h,2w,2) | None, idx int32 | None)."""
    n, hl, wl, _ = flow_lo.shape
    H, W = 2 * hl, 2 * wl
    assert dst.h == H and dst.w == W
    dev = flow_lo.device
    flow_up = torch.empty((n, H, W, 2), dtype=torch.float32, device=dev) if want_flow_up else None
    idx = torch.empty((n, H, W, 2), dtype=torch.int32, device=dev) if want_idx else None
    ts, td = src.ct(), dst.ct()
    with _Timed("glue", 0.0, label="flow_warp"):
        capi.check(_L(src, dst).hrv_flow_warp(flow_lo.data_ptr(), linspace_table(W, dev).data_ptr(), linspace_table(H, dev).data_ptr(),
                                            ctypes.byref(ts), ctypes.byref(td), _p(flow_up), _p(idx), _stream()), "flow_warp")
    return flow_up, idx


def norm_bwd(dh, h, gamma, x0, x0_shift, x1, noise, noise_scale, mean, rstd, act, want_dgb, chan_scale=None, batch_stats=False):
    """Fused backward of the SPADE modulation + InstanceNorm (gamma given) or of InstanceNorm + activation (gamma None).
    Returns (dgb Act | None, dx0 Act, dx1 Act | None, d_noise_scale fp32 [C] | None, sum_dgamma fp32 [C], sum_dbeta fp32 [C])."""
    n, H, W = dh.n, dh.h, dh.w
    c0 = x0.c
    c1 = x1.c if x1 is not None else 0
    C = c0 + c1
    dev = dh.buf.device
    dxn = Act.empty(n, H, W, C)
    dgb = Act.empty(n, H, W, 2 * C) if want_dgb else None
    sums = torch.empty((n, C, 4), dtype=torch.float64, device=dev)
    tdh, tx0, tdxn = dh.ct(), x0.ct(), dxn.ct()
    th = h.ct() if h is not None else _NULL
    tg = gamma.ct() if gamma is not None else _NULL
    tx1 = x1.ct() if x1 is not None else _NULL
    tdgb = dgb.ct() if dgb is not None else _NULL
    with _Timed("norm_bwd", n * H * W * C * 2.0 * (4 + (1 if gamma is not None else 0) + (2 if want_dgb else 0)), launches=2):
        capi.check(_L(dh).hrv_norm_bwd_reduce(ctypes.byref(tdh), ctypes.byref(th), ctypes.byref(tg), ctypes.byref(tx0), x0_shift,
                                                  ctypes.byref(tx1), H, W, _p(noise), _p(noise_scale), mean.data_ptr(), rstd.data_ptr(),
                                                  _p(chan_scale), act, ctypes.byref(tdgb), ctypes.byref(tdxn), sums.data_ptr(), _stream()), "norm_bwd_reduce")
    if batch_stats:  # BatchNorm: the two means run over (N,H,W)
        tot = sums.sum(0, keepdim=True) / float(n * H * W)
        m1 = tot[:, :, 0].expand(n, C).float().contiguous()
        m2 = tot[:, :, 1].expand(n, C).float().contiguous()
    else:
        inv = 1.0 / float(H * W)
        m1 = (sums[:, :, 0] * inv).float().contiguous()
        m2 = (sums[:, :, 1] * inv).float().contiguous()
    dns = torch.zeros(C, dtype=torch.float64, device=dev) if noise_scale is not None else None
    dx0 = Act.empty(n, x0.h, x0.w, c0)
    tdx0 = dx0.ct()
    with _Timed("norm_bwd", n * H * W * c0 * 2.0 * 2, launches=1):
        capi.check(_L(dh).hrv_norm_bwd_apply(ctypes.byref(tdxn), ctypes.byref(tx0), x0_shift, 0, C, H, W, _p(noise), _p(noise_scale),
                                                 mean.data_ptr(), rstd.data_ptr(), m1.data_ptr(), m2.data_ptr(), ctypes.byref(tdx0),
                                                 _p(dns), _stream()), "norm_bwd_apply(x0)")
    dx1 = None
    if x1 is not None:
        dx1 = Act.empty(n, H, W, c1)
        tdx1 = dx1.ct()
        with _Timed("norm_bwd", n * H * W * c1 * 2.0 * 3, launches=1):
            capi.check(_L(dh).hrv_norm_bwd_apply(ctypes.byref(tdxn), ctypes.byref(tx1), 0, c0, C, H, W, _p(noise), _p(noise_scale),
                                                     mean.data_ptr(), rstd.data_ptr(), m1.data_ptr(), m2.data_ptr(), ctypes.byref(tdx1),
                                                     _p(dns), _stream()), "norm_bwd_apply(x1)")
    return dgb, dx0, dx1, (dns.float() if dns is not None else None), sums[:, :, 2].sum(0).float(), sums[:, :, 3].sum(0).float()


def act_bwd_bias(dy, y, act, want_dv=True, want_bias=True):
    """(dv Act | dy itself when act is NONE, bias_grad fp32 [c] | None) for an epilogue act(conv + b)."""
    c8 = round_up(dy.c, 8)
    dv = Act.empty(dy.n, dy.h, dy.w, dy.c, pitch=dy.pitch) if (want_dv and act != ACT_NONE) else None
    bsum = torch.empty(c8, dtype=torch.float64, device=dy.buf.device) if want_bias else None
    if dv is None and bsum is None:
        return dy, None
    tdy = dy.ct()
    ty = y.ct() if (y is not None and act != ACT_NONE) else _NULL
    tdv = dv.ct() if dv is not None else _NULL
    with _Timed("act_bwd", dy.n * dy.h * dy.w * dy.c * 2.0 * (3 if dv is not None else 1)):
        capi.check(_L(dy).hrv_act_bwd_bias(ctypes.byref(tdy), ctypes.byref(ty), act, ctypes.byref(tdv), _p(bsum), _stream()), "act_bwd_bias")
    return (dv if dv is not None else dy), (bsum[:dy.c].float() if bsum is not None else None)


def conv2d_wgrad(x, dy, kh, kw, pad):
    """dW (cout,cin,kh,kw) fp32 of a stride-1 convolution, on tcgen05 (hrv_conv2d_wgrad)."""
    dw = torch.empty((dy.c, x.c, kh, kw), dtype=torch.float32, device=x.buf.device)
    tx, tdy = x.ct(), dy.ct()
    L = _L(x)
    nws = int(L.hrv_conv2d_wgrad_workspace_bytes(ctypes.byref(tx), ctypes.byref(tdy), kh, kw))
    ws = torch.empty(nws, dtype=torch.uint8, device=x.buf.device) if nws else None  # split-K slabs, summed in a fixed order (deterministic)
    with _Timed("wgrad", 2.0 * x.c * dy.c * kh * kw * dy.n * dy.h * dy.w, launches=2 if nws else 1,
                label="%d->%d k%dx%d n%d %dx%d" % (x.c, dy.c, kh, kw, dy.n, dy.h, dy.w)):
        capi.check(L.hrv_conv2d_wgrad(ctypes.byref(tx), ctypes.byref(tdy), kh, kw, pad, dw.data_ptr(), _p(ws), nws, _stream()), "conv2d_wgrad")
    return dw


def batchnorm_stats(x, eps=1e-5):
    """Train-mode BatchNorm2d statistics over (N,H,W) from ONE pass of the statistics kernel (per-image fp64 partial sums combined
    here on [N][C] scalars) — the "single-kernel reduce" standing in for SyncBatchNorm.  Returns (mean[C], biased var[C]) fp32."""
    n, c = x.n, x.c
    ws = _workspace(n * c * 16, x.buf.device)
    mean_nc = torch.empty((n, c), dtype=torch.float32, device=x.buf.device)
    rstd_nc = torch.empty_like(mean_nc)
    t0 = x.ct()
    with _Timed("instnorm_stats", n * x.h * x.w * 2.0 * c, launches=3, label="bn c%d n%d %dx%d" % (c, n, x.h, x.w)):
        capi.check(_L(x).hrv_instnorm_stats(ctypes.byref(t0), 0, ctypes.byref(_NULL), x.h, x.w, None, None, eps, mean_nc.data_ptr(),
                                                 rstd_nc.data_ptr(), ws.data_ptr(), ws.numel(), _stream()), "batchnorm_stats")
    sums = ws[: n * c * 16].view(torch.float64).view(n, c, 2).sum(0)  # raw sum / sum of squares left in the workspace
    cnt = float(n * x.h * x.w)
    mean = sums[:, 0] / cnt
    var = (sums[:, 1] / cnt - mean * mean).clamp_min(0.0)
    return mean.float(), var.float()


def norm_apply_affine(x, mean_nc, rstd_nc, gamma, beta, res, act, out=None):
    out = Act.empty(x.n, x.h, x.w, x.c) if out is None else out
    tx, ty = x.ct(), out.ct()
    tr = res.ct() if res is not None else _NULL
    with _Timed("norm_apply", x.n * x.h * x.w * x.c * 2.0 * (3 if res is not None else 2)):
        capi.check(_L(x).hrv_norm_apply_affine(ctypes.byref(tx), mean_nc.data_ptr(), rstd_nc.data_ptr(), _p(gamma), _p(beta),
                                                    ctypes.byref(tr), act, ctypes.byref(ty), _stream()), "norm_apply_affine")
    return out


def bilinear_up2_bwd(dout):
    da = Act.empty(dout.n, dout.h // 2, dout.w // 2, dout.c)
    td, ta = dout.ct(), da.ct()
    with _Timed("up2_bwd", dout.n * dout.h * dout.w * dout.c * 2.0 * 1.25):
        capi.check(_L(dout).hrv_bilinear_up2_bwd(ctypes.byref(td), ctypes.byref(ta), _stream()), "bilinear_up2_bwd")
    return da


def flow_warp_bwd(flow_lo, src, ddst, dflow_up_in, want_dsrc=True):
    """Returns (dsrc bf16 Act | None, dflow_lo fp32 (N,h,w,2))."""
    n, hl, wl, _ = flow_lo.shape
    H, W = 2 * hl, 2 * wl
    dev = flow_lo.device
    c8 = round_up(src.c, 8)
    dsrc32 = torch.zeros((n, src.h, src.w, c8), dtype=torch.float32, device=dev) if want_dsrc else None
    dfu = dflow_up_in.float().contiguous().clone() if dflow_up_in is not None else torch.zeros((n, H, W, 2), dtype=torch.float32, device=dev)
    dflo = torch.empty((n, hl, wl, 2), dtype=torch.float32, device=dev)
    ts, td = src.ct(), ddst.ct()
    with _Timed("flow_warp_bwd", n * H * W * src.c * 2.0 * 3, launches=2):
        capi.check(_L(src, ddst).hrv_flow_warp_bwd(flow_lo.data_ptr(), linspace_table(W, dev).data_ptr(), linspace_table(H, dev).data_ptr(),
                                                ctypes.byref(ts), ctypes.byref(td), _p(dsrc32), dfu.data_ptr(), dflo.data_ptr(), _stream()),
                   "flow_warp_bwd")
    dsrc = Act(dsrc32.to(src.buf.dtype)) if want_dsrc else None
    return dsrc, dflo
