import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hrv_loader; hrv_loader.load()
from hrviton_b200 import ops
from hrviton_b200.ops import Act
torch.manual_seed(0)
def run(spade, cin, ng, h, w, B, pair, shift=0, c1=0):
    os.environ["HRV_CONV_PAIR"] = "1" if pair else "0"
    os.environ["HRV_CONV_PIXN"] = "0"
    x = Act(torch.randn(B, h, w, ops.round_up(cin, 8), device="cuda").to(torch.bfloat16), c=cin)
    if spade:
        C = ng // 2
        wt = torch.randn(C, cin, 3, 3, device="cuda") * 0.05; wt2 = torch.randn(C, cin, 3, 3, device="cuda") * 0.05
        pw = ops.pack_weight(wt, (1, 1), interleave=wt2)
        x0 = Act(torch.randn(B, h >> shift, w >> shift, C - c1, device="cuda").to(torch.bfloat16))
        x1 = Act(torch.randn(B, h, w, c1, device="cuda").to(torch.bfloat16)) if c1 else None
        mean = torch.randn(B, C, device="cuda") * 0.1; rstd = torch.rand(B, C, device="cuda") + 0.5
        noise = torch.randn(B, h, w, device="cuda"); ns = torch.randn(C, device="cuda") * 0.1; sh = torch.randn(2 * C, device="cuda") * 0.1
        out = Act.empty(B, h, w, C); gam = Act.empty(B, h, w, C)
        ops.conv2d_spade(x, pw, out, x0, shift, x1, mean, rstd, noise, ns, sh, 2, gamma_out=gam)
        torch.cuda.synchronize()
        return out.buf.float().clone(), gam.buf.float().clone()
    wt = torch.randn(ng, cin, 3, 3, device="cuda") * 0.05
    pw = ops.pack_weight(wt, (1, 1))
    out = Act.empty(B, h, w, ng)
    ops.conv2d(x, pw, out, act=2, shift=torch.randn(ng, device="cuda"))
    torch.cuda.synchronize()
    return out.buf.float().clone(), None
for spade, cin, ng, h, w, B, shift, c1 in [(True, 128, 160, 64, 48, 2, 0, 0), (True, 128, 288, 40, 24, 1, 0, 0), (False, 160, 160, 50, 37, 3, 0, 0),
                                         (True, 128, 544, 32, 24, 2, 0, 0), (False, 80, 192, 128, 96, 1, 0, 0), (True, 128, 160, 64, 48, 2, 1, 16),
                                         (True, 128, 288, 48, 32, 3, 1, 16), (True, 128, 544, 32, 24, 1, 1, 16), (True, 128, 2080, 16, 12, 2, 1, 16),
                                         (False, 256, 256, 40, 30, 2, 0, 0), (True, 128, 144, 30, 22, 1, 0, 0),
                                         # many items per CTA pair with 2 TMEM accumulators (3 epilogue warpgroups, 2 owners) and with 3
                                         (True, 128, 544, 256, 192, 2, 1, 16), (False, 256, 256, 256, 192, 2, 0, 0), (True, 128, 160, 512, 384, 2, 1, 16)]:
    torch.manual_seed(1); a, ga = run(spade, cin, ng, h, w, B, False, shift, c1)
    torch.manual_seed(1); b, gb = run(spade, cin, ng, h, w, B, True, shift, c1)
    d = float((a - b).abs().max()); print("pair vs single", spade, cin, ng, h, w, B, shift, c1, "max diff", d, "gamma", float((ga - gb).abs().max()) if ga is not None else None, flush=True)
    halo_single = spade or ng <= 208  # the one-CTA kernel walks K in the same (chunk, tap) order only in its halo mainloop
    assert d == 0.0 if halo_single else d <= 2 ** -7 * float(a.abs().max()), (d, float(a.abs().max()))
print("PAIR OK")
