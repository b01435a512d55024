"""GPU: gradient parity of the training path (hrviton_b200.autograd_g / autograd_tocg) against torch autograd run through the
CPU oracle (fp32) on identical weights / inputs / noise.  Bounds are derived, not hand-picked: the same oracle is re-run with its
convolutions rounding to bf16 (oracle.storage_rounding, gradients rounded at the same points) and the kernels' per-parameter
relative L2 errors must stay within 1.1 x that floor in median / p90 (floors.RATIO_MAX in max; 1.6-2 x per individual parameter)."""
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "oracle"))
import hrviton_oracle as orc  # noqa: E402
from helpers import gen_opt, synth_state_dict  # noqa: E402
from hrviton_b200 import synth  # noqa: E402

pytestmark = pytest.mark.gpu


def _oracle_gen_grads(sd, x, seg, R, seed, rounding=None, sn_train=False):
    """(out, {name: grad}, state after the forward) of the oracle generator, loss = sum(out * R); optional storage rounding model."""
    sdr = {k: v.clone().requires_grad_(v.is_floating_point() and not k.endswith(("weight_u", "weight_v"))) for k, v in sd.items()}
    cnt = [0]

    def noise_cpu(b, hh, ww):
        t = synth.spade_noise(b, hh, ww, seed, cnt[0])
        cnt[0] += 1
        return t

    import contextlib
    with orc.storage_rounding(rounding), (orc.spectral_train() if sn_train else contextlib.nullcontext()):
        out = orc.spade_generator_forward(sdr, x, seg, noise_cpu)
    (out * R).sum().backward()
    return out.detach(), {k: v.grad for k, v in sdr.items() if v.requires_grad and v.grad is not None}, sdr


def _rel_rows(grads_got, grads_ref):
    rows = {}
    for name, gr in grads_ref.items():
        g = grads_got[name].detach().float().cpu()
        nref = float(gr.norm())
        rows[name] = (float((g - gr).norm()) / (nref + 1e-12), float((g * gr).sum() / (g.norm() * gr.norm() + 1e-20)), nref, float(g.norm()))
    return rows


def _check_against_floor(tag, rows, floor_rows, gmax, per_param_ratio=1.6):
    """Kernel gradient errors vs the storage-rounded oracle's own errors (both against fp32 oracle autograd).
    Aggregate statistics carry the 1.1x bound; individual parameters (each a different realisation of the rounding noise) 1.6x."""
    import floors
    live = [n for n, r in floor_rows.items() if r[2] > 1e-5 * gmax]
    dead = [n for n in floor_rows if n not in live]
    for n in dead:  # mathematically zero gradients (biases feeding an InstanceNorm): ours must be negligible too
        assert rows[n][3] < 2e-2 * gmax, "%s should have ~zero gradient, got %.3e (max grad norm %.3e)" % (n, rows[n][3], gmax)
    mine = sorted(rows[n][0] for n in live)
    flo = sorted(floor_rows[n][0] for n in live)
    q = lambda v, f: v[min(len(v) - 1, int(len(v) * f))]
    print("GRADPARITY %s: %d live / %d zero-gradient parameters | kernels median %.3e p90 %.3e max %.3e | rounded-oracle floor median %.3e p90 %.3e max %.3e"
          % (tag, len(live), len(dead), q(mine, 0.5), q(mine, 0.9), mine[-1], q(flo, 0.5), q(flo, 0.9), flo[-1]))
    worst = sorted(((rows[n][0] / max(floor_rows[n][0], 1e-9), n) for n in live), reverse=True)[:5]
    for ratio, n in worst:
        print("GRADPARITY %s worst ratio x%.2f  ours %.3e floor %.3e cos %.5f  %s" % (tag, ratio, rows[n][0], floor_rows[n][0], rows[n][1], n))
    assert q(mine, 0.5) <= floors.RATIO * q(flo, 0.5)
    assert q(mine, 0.9) <= floors.RATIO * q(flo, 0.9)
    assert mine[-1] <= floors.RATIO_MAX * flo[-1]
    cos_mine, cos_flo = min(rows[n][1] for n in live), min(floor_rows[n][1] for n in live)
    print("GRADPARITY %s: worst cosine kernels %.5f, rounded oracle %.5f" % (tag, cos_mine, cos_flo))
    assert (1.0 - cos_mine) <= floors.RATIO_MAX * (1.0 - cos_flo) + 1e-3
    for n in live:
        assert rows[n][0] <= per_param_ratio * floor_rows[n][0] + 5e-3, (n, rows[n][0], floor_rows[n][0])
    return mine, flo


@pytest.mark.parametrize("sn_train", [False, True], ids=["eval_sn", "train_sn"])
def test_generator_gradients(sn_train):
    """Generator forward + backward vs fp32 oracle autograd.  train_sn: the module is in train() mode, i.e. spectral norm runs its
    power iteration (u, v refreshed in place, gradient through sigma = u.(W v)) — buffers and gradients are compared with the
    oracle's train-mode restatement (network_generator.py:138-143)."""
    import network_generator
    n, h, w, seed = (1, 512, 384, 23) if not sn_train else (1, 256, 256, 29)
    sd = synth_state_dict("gen", seed)
    x, seg = synth.gen_inputs(n, h, w, seed)
    R = synth.normalish((n, 3, h, w), seed, "lossw")
    out_ref, g_ref, sd_after = _oracle_gen_grads(sd, x, seg, R, seed, None, sn_train)
    out_flo, g_flo, _ = _oracle_gen_grads(sd, x, seg, R, seed, torch.bfloat16, sn_train)
    floor_rows = _rel_rows(g_flo, g_ref)
    # ---- product path
    m = network_generator.SPADEGenerator(gen_opt(h, w, True), 9)
    m.load_state_dict(sd)
    m = m.cuda()
    m.train(sn_train)
    cnt2 = [0]

    def noise_dev(b, hh, ww):
        t = synth.spade_noise(b, hh, ww, seed, cnt2[0]).cuda()
        cnt2[0] += 1
        return t

    m.noise_source = noise_dev
    out = m(x.cuda(), seg.cuda())
    assert out.requires_grad
    (out * R.cuda()).sum().backward()
    torch.cuda.synchronize()
    import floors
    floors.check("gen train fwd (sn_train=%s)" % sn_train, out.detach(), out_ref.numpy(), floors.stats(out_flo, out_ref.numpy()))
    if sn_train:  # power iteration: u, v after the forward equal torch's (fp32 gemv both sides)
        after = m.state_dict()
        for k in [k for k in sd if k.endswith(("weight_u", "weight_v"))]:
            assert not torch.equal(sd[k], sd_after[k].detach()), k  # the oracle moved them ...
            d = float((after[k].cpu() - sd_after[k].detach()).abs().max())
            assert d < 1e-4, (k, d)                                   # ... and the module moved them identically
    grads = {name: p.grad for name, p in m.named_parameters() if p.grad is not None}
    for name in g_ref:
        assert name in grads, name
    rows = _rel_rows(grads, g_ref)
    gmax = max(r[2] for r in rows.values())
    for name, (rel, cos, nref, ng) in rows.items():
        print("GRADPARITY %-44s ref %.3e got %.3e rel %.3e floor %.3e cos %.5f" % (name, nref, ng, rel, floor_rows[name][0], cos))
    _check_against_floor("generator sn_train=%s" % sn_train, rows, floor_rows, gmax)
    # the last layer sees no accumulated rounding: it must be tight in absolute terms, not only relative to the floor
    assert rows["conv_img.weight"][0] < 3e-2 and rows["conv_img.bias"][0] < 1e-2
    assert rows["up_4.norm_0.noise_scale"][2] > 0  # the noise-scale parameters are on the checked path


def _d_loss(res):
    return sum((f * (1 + 0.1 * j)).mean() for fs in res for j, f in enumerate(fs))


def _oracle_d_grads(fwd, sd, inp, rounding=None):
    sdr = {k: v.clone().requires_grad_(v.is_floating_point() and not k.endswith(("weight_u", "weight_v"))) for k, v in sd.items()}
    inp_ref = inp.clone().requires_grad_(True)
    with orc.storage_rounding(rounding):
        res = fwd(sdr, inp_ref)
    _d_loss(res).backward()
    grads = {k: v.grad for k, v in sdr.items() if v.requires_grad and v.grad is not None and float(v.grad.norm()) > 1e-7}
    grads["__input__"] = inp_ref.grad
    return [[f.detach() for f in fs] for fs in res], grads


def _check_d(tag, res, res_ref, res_flo, grads, g_ref, g_flo):
    import floors
    for i, fs in enumerate(res):
        for j, f in enumerate(fs):
            floors.check("%s d%d_f%d" % (tag, i, j), f.detach(), res_ref[i][j].numpy(), floors.stats(res_flo[i][j], res_ref[i][j].numpy()),
                         extra_abs=1e-4)
    rows, floor_rows = _rel_rows(grads, g_ref), _rel_rows(g_flo, g_ref)
    print("GRADPARITY %s input gradient rel %.3e (floor %.3e)" % (tag, rows["__input__"][0], floor_rows["__input__"][0]))
    gmax = max(r[2] for r in rows.values())
    _check_against_floor(tag, rows, floor_rows, gmax, per_param_ratio=2.0)  # tiny maps (9x7 .. 33x25): few samples per parameter


def test_discriminator_gradients():
    """gen-D training path: gradient w.r.t. the input image and all parameters vs torch autograd through the oracle; bounds =
    1.1 x the bf16-rounded oracle's own deviation."""
    import network_generator
    from hrviton_b200 import autograd_g
    n, h, w, seed = 2, 128, 96, 31
    sd = synth_state_dict("gend", seed)
    x, seg = synth.gen_inputs(n, h, w, seed, input_nc=3)
    inp = torch.cat([seg, x], 1)
    res_ref, g_ref = _oracle_d_grads(orc.gen_d_forward, sd, inp)
    res_flo, g_flo = _oracle_d_grads(orc.gen_d_forward, sd, inp, torch.bfloat16)
    m = network_generator.MultiscaleDiscriminator(gen_opt(h, w, True))
    m.load_state_dict(sd)
    m = m.cuda().eval()
    inp_d = inp.cuda().requires_grad_(True)
    res = autograd_g.discriminator_forward_train(m, inp_d, need_wgrad=True)
    _d_loss(res).backward()
    torch.cuda.synchronize()
    grads = {name: p.grad for name, p in m.named_parameters() if p.grad is not None}
    grads["__input__"] = inp_d.grad
    _check_d("gen-D", res, res_ref, res_flo, grads, g_ref, g_flo)


def test_tocg_discriminator_gradients():
    """Stage-1 discriminator (networks.define_D, LSGAN PatchGAN with InstanceNorm, Ddownx2) through the MODULE's own forward in
    train mode with grad enabled — the call train_condition.py:208-232 makes — vs oracle autograd (dropout off: it is torch's
    RNG in the reference too and cannot be replayed)."""
    import contextlib
    import io

    import networks
    seed = 37
    with contextlib.redirect_stdout(io.StringIO()):
        m = networks.define_D(input_nc=33, Ddownx2=True, Ddropout=False, n_layers_D=3, spectral=False, num_D=2)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    synth.fill_state_dict(sd, seed)
    m.load_state_dict(sd)
    m = m.cuda().train()
    i1, i2 = synth.tocg_inputs(1, 256, 192, seed)
    segs = synth.one_hot(synth.labels((1, 256, 192), 13, seed, "dseg"), 13)
    inp = torch.cat([i1, i2, segs], 1)
    res_ref, g_ref = _oracle_d_grads(orc.tocg_d_forward, sd, inp)
    res_flo, g_flo = _oracle_d_grads(orc.tocg_d_forward, sd, inp, torch.bfloat16)
    inp_d = inp.cuda().requires_grad_(True)
    res = m(inp_d)  # dispatches to the autograd path
    assert res[0][0].requires_grad
    _d_loss(res).backward()
    torch.cuda.synchronize()
    grads = {name: p.grad for name, p in m.named_parameters() if p.grad is not None}
    grads["__input__"] = inp_d.grad
    _check_d("tocg-D", res, res_ref, res_flo, grads, g_ref, g_flo)


def test_tocg_discriminator_intermediate_features_are_differentiable():
    """Stage-1 discriminator with getIntermFeat=True in train mode with grad enabled: every per-layer feature carries a gradient, and
    the same layers, split into one sequence per layer group, compute what the flat getIntermFeat=False discriminator computes — the
    logits and the weight gradients bit for bit."""
    import contextlib
    import io

    import networks
    seed = 37
    with contextlib.redirect_stdout(io.StringIO()):
        flat = networks.define_D(input_nc=33, Ddownx2=True, Ddropout=False, n_layers_D=3, spectral=False, num_D=2)
        inter = networks.define_D(input_nc=33, Ddownx2=True, Ddropout=False, n_layers_D=3, spectral=False, num_D=2, getIntermFeat=True)
    sd = {k: v.clone() for k, v in flat.state_dict().items()}
    synth.fill_state_dict(sd, seed)
    flat.load_state_dict(sd)
    inter_keys = list(inter.state_dict())
    assert len(inter_keys) == len(sd)
    inter.load_state_dict(dict(zip(inter_keys, sd.values())))  # same layers in the same order: the keys map one to one
    flat, inter = flat.cuda().train(), inter.cuda().train()
    i1, i2 = synth.tocg_inputs(1, 256, 192, seed)
    segs = synth.one_hot(synth.labels((1, 256, 192), 13, seed, "dseg"), 13)
    inp = torch.cat([i1, i2, segs], 1).cuda()
    res_flat, res_inter = flat(inp), inter(inp)
    assert len(res_inter) == 2 and all(len(fs) == 5 for fs in res_inter)
    assert all(f.requires_grad for fs in res_inter for f in fs)
    for fs, (logits,) in zip(res_inter, res_flat):
        assert torch.equal(fs[-1], logits)
    for res in (res_flat, res_inter):
        sum((fs[-1] * fs[-1]).mean() for fs in res).backward()
    torch.cuda.synchronize()
    for (name, p), (name_i, p_i) in zip(flat.named_parameters(), inter.named_parameters()):
        assert p.grad is not None and torch.equal(p.grad, p_i.grad), (name, name_i)


def test_stage2_train_step_runs():
    """One full stage-2 step (tocg -> warp -> G -> D -> hinge/feat/VGG -> Adam x2) at 512x384: finite losses, parameters move."""
    import types

    import network_generator
    import networks
    from hrviton_b200 import train_step
    os.environ["HRV_VGG_RANDOM_INIT"] = "1"
    h, w = 512, 384
    topt = types.SimpleNamespace(warp_feature="T1", out_layer="relu", cuda=True)
    tocg = networks.ConditionGenerator(topt, 4, 16, 13, ngf=96, norm_layer=torch.nn.BatchNorm2d)
    sdt = tocg.state_dict()
    synth.fill_state_dict(sdt, 3)
    tocg.load_state_dict(sdt)
    tocg = tocg.cuda().eval()
    G = network_generator.SPADEGenerator(gen_opt(h, w, True), 9)
    sdg = G.state_dict()
    synth.fill_state_dict(sdg, 4)
    G.load_state_dict(sdg)
    G = G.cuda().train()
    D = network_generator.MultiscaleDiscriminator(gen_opt(h, w, True))
    sdd = D.state_dict()
    synth.fill_state_dict(sdd, 5)
    D.load_state_dict(sdd)
    D = D.cuda().train()
    vgg = networks.Vgg19().cuda().eval()
    tr = train_step.Stage2Trainer(tocg, G, D, vgg)
    batch = train_step.synthetic_batch(1, h, w, "cuda", seed=7)
    w_before = G.up_3.conv_0.weight_orig.detach().clone()
    d_before = D.discriminator_0.model0[0].weight.detach().clone()
    out = tr.step(batch, h, w)
    torch.cuda.synchronize()
    print("TRAINSTEP losses:", {k: float(v) for k, v in out.items()})
    assert all(torch.isfinite(torch.as_tensor(float(v))) for v in out.values())
    assert float((G.up_3.conv_0.weight_orig.detach() - w_before).abs().max()) > 0
    assert float((D.discriminator_0.model0[0].weight.detach() - d_before).abs().max()) > 0


def _oracle_tocg_train(sd, i1, i2, Rs, Rc, rounding=None):
    sdr = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else v.clone()) for k, v in sd.items()}
    with orc.storage_rounding(rounding):
        flows_r, seg_r, wc_r, wcm_r = orc.tocg_forward(sdr, i1, i2, bn_train=True)
    (seg_r * Rs).mean().add((wc_r * Rc).mean()).add(sum(f.abs().mean() for f in flows_r)).backward()
    grads = {k: v.grad for k, v in sdr.items() if torch.is_tensor(v) and v.requires_grad and v.grad is not None and float(v.grad.norm()) > 1e-7}
    return [f.detach() for f in flows_r], seg_r.detach(), wc_r.detach(), grads


def test_tocg_training_gradients():
    """Condition generator in train mode through the MODULE's forward (the call train_condition.py:158 makes): batch-statistics
    BatchNorm (statistics kernel + fused backward), outputs and parameter gradients vs torch autograd through the oracle with
    bn_train=True; bounds = 1.1 x the bf16-rounded oracle's own deviation (train-mode BatchNorm over as few as 4x3x2 samples is
    ~10x more sensitive to storage rounding than eval mode — for the fp32 algorithm itself)."""
    import floors
    import networks
    from helpers import tocg_opt
    n, h, w, seed = 2, 256, 192, 11
    sd = synth_state_dict("tocg", seed)
    i1, i2 = synth.tocg_inputs(n, h, w, seed)
    Rs = synth.normalish((n, 13, h, w), seed, "rs")
    Rc = synth.normalish((n, 3, h, w), seed, "rc")
    flows_r, seg_r, wc_r, g_ref = _oracle_tocg_train(sd, i1, i2, Rs, Rc)
    flows_f, seg_f, wc_f, g_flo = _oracle_tocg_train(sd, i1, i2, Rs, Rc, torch.bfloat16)
    m = networks.ConditionGenerator(tocg_opt(True), 4, 16, 13, ngf=96, norm_layer=torch.nn.BatchNorm2d)
    m.load_state_dict(sd)
    m = m.cuda().train()
    flows, seg, wc, wcm = m(i1.cuda(), i2.cuda())  # train mode: forward() dispatches to the differentiable path
    assert seg.requires_grad
    ((seg * Rs.cuda()).mean() + (wc * Rc.cuda()).mean() + sum(f.abs().mean() for f in flows)).backward()
    torch.cuda.synchronize()
    floors.check("tocg train seg", seg.detach(), seg_r.numpy(), floors.stats(seg_f, seg_r.numpy()))
    floors.check("tocg train flow4", flows[-1].detach(), flows_r[-1].numpy(), floors.stats(flows_f[-1], flows_r[-1].numpy()))
    floors.check("tocg train warped_c", wc.detach(), wc_r.numpy(), floors.stats(wc_f, wc_r.numpy()))
    # running statistics must have moved exactly as torch's BatchNorm2d would move them (momentum 0.1)
    bn = m.ClothEncoder[0].block[1]
    assert int(bn.num_batches_tracked) == 1
    grads = {name: p.grad for name, p in m.named_parameters() if p.grad is not None}
    rows, floor_rows = _rel_rows({k: grads[k] for k in g_ref}, g_ref), _rel_rows({k: g_flo[k] for k in g_ref if k in g_flo}, {k: g_ref[k] for k in g_ref if k in g_flo})
    rows = {k: rows[k] for k in floor_rows}
    gmax = max(r[2] for r in rows.values())
    _check_against_floor("tocg train", rows, floor_rows, gmax, per_param_ratio=2.0)
    assert m.conv2[0].weight.grad is None  # dead branch of the reference (networks.py:131)


def test_stage1_train_step_runs():
    """One full stage-1 step (tocg fwd+bwd with train-mode BN, tocg-D x3, L1 + VGG x5 + TV + CE + LSGAN, Adam x2) at 256x192."""
    import contextlib
    import io

    import networks
    from helpers import tocg_opt
    from hrviton_b200 import train_step
    os.environ["HRV_VGG_RANDOM_INIT"] = "1"
    tocg = networks.ConditionGenerator(tocg_opt(True), 4, 16, 13, ngf=96, norm_layer=torch.nn.BatchNorm2d)
    sdt = tocg.state_dict()
    synth.fill_state_dict(sdt, 3)
    tocg.load_state_dict(sdt)
    tocg = tocg.cuda().train()
    with contextlib.redirect_stdout(io.StringIO()):
        D = networks.define_D(input_nc=33, Ddownx2=True, Ddropout=True, n_layers_D=3, spectral=False, num_D=2)
    D = D.cuda().train()
    vgg = networks.Vgg19().cuda().eval()
    tr = train_step.Stage1Trainer(tocg, D, vgg)
    batch = train_step.synthetic_batch_stage1(2, 256, 192, "cuda", seed=9)
    w_before = tocg.flow_conv[4].weight.detach().clone()
    d_before = D.layer0[0].weight.detach().clone()
    out = tr.step(batch)
    torch.cuda.synchronize()
    print("TRAINSTEP1 losses:", {k: float(v) for k, v in out.items()})
    assert all(torch.isfinite(torch.as_tensor(float(v))) for v in out.values())
    assert float((tocg.flow_conv[4].weight.detach() - w_before).abs().max()) > 0
    assert float((D.layer0[0].weight.detach() - d_before).abs().max()) > 0
    assert tocg.conv2[0].weight.grad is None  # dead branch of the reference (networks.py:131) receives no gradient


def test_stage2_losses_match_oracle_pipeline():
    """The measured workload itself: generator-update losses of Stage2Trainer (tocg -> glue -> G -> D -> hinge/feature-matching/VGG)
    against the same pipeline evaluated with the CPU oracle networks (fp32) on identical weights, batch and SPADE noise."""
    import types

    import network_generator
    import networks
    import torch.nn.functional as F
    from hrviton_b200 import autograd_g, train_step
    os.environ["HRV_VGG_RANDOM_INIT"] = "1"
    h = w = 256
    n = 1
    seed = 17
    topt = types.SimpleNamespace(warp_feature="T1", out_layer="relu", cuda=True)
    tocg = networks.ConditionGenerator(topt, 4, 16, 13, ngf=96, norm_layer=torch.nn.BatchNorm2d)
    sdt = tocg.state_dict(); synth.fill_state_dict(sdt, seed); tocg.load_state_dict(sdt)
    G = network_generator.SPADEGenerator(gen_opt(h, w, True), 9)
    sdg = G.state_dict(); synth.fill_state_dict(sdg, seed + 1); G.load_state_dict(sdg)
    D = network_generator.MultiscaleDiscriminator(gen_opt(h, w, True))
    sdd = D.state_dict(); synth.fill_state_dict(sdd, seed + 2); D.load_state_dict(sdd)
    torch.manual_seed(0)
    vgg = networks.Vgg19()
    vgg_cpu_sd = {k: v.clone() for k, v in vgg.state_dict().items()}
    tocg, G, D, vgg = tocg.cuda().eval(), G.cuda().eval(), D.cuda().eval(), vgg.cuda().eval()
    batch = train_step.synthetic_batch(n, h, w, "cpu", seed=seed)
    cnt = [0]

    def noise_dev(b, hh, ww):
        t = synth.spade_noise(b, hh, ww, seed, cnt[0]).cuda()
        cnt[0] += 1
        return t

    G.noise_source = noise_dev
    # ---- product path (forward part of Stage2Trainer.step, generator update)
    bd = {k: v.cuda() for k, v in batch.items()}
    with torch.no_grad():
        g_in, parse = train_step.make_generator_inputs(tocg, bd, h, w, occlusion=True)  # the README's --occlusion configuration
        out = G(g_in, parse)
        d_in = torch.cat((torch.cat((parse, out), 1), torch.cat((parse, bd["image"]), 1)), 0)
        pred = autograd_g.discriminator_forward_train(D, d_in, need_wgrad=False, as_float=True)
        fake = [[t[:n] for t in p] for p in pred]
        real = [[t[n:] for t in p] for p in pred]
        crit = network_generator.GANLoss("hinge")
        gan = float(crit(fake, True, for_discriminator=False))
        feat = float(sum(F.l1_loss(fake[i][j], real[i][j]) * 10.0 / 2 for i in range(2) for j in range(len(fake[i]) - 1)))
        vl = float(autograd_g.vgg_loss(vgg, [1.0 / 32, 1.0 / 16, 1.0 / 8, 1.0 / 4, 1.0], out, bd["image"]))
    # ---- oracle pipeline on the CPU (same glue code, oracle networks)
    class _OracleTocg:
        def __call__(self, i1, i2):
            return orc.tocg_forward(sdt, i1, i2)
    c2 = [0]

    def noise_cpu(b, hh, ww):
        t = synth.spade_noise(b, hh, ww, seed, c2[0])
        c2[0] += 1
        return t

    with torch.no_grad():
        g_in_r, parse_r = train_step.make_generator_inputs(_OracleTocg(), batch, h, w, unfused_parse=True, occlusion=True)
        out_r = orc.spade_generator_forward(sdg, g_in_r, parse_r, noise_cpu)
        pred_r = orc.gen_d_forward(sdd, torch.cat((torch.cat((parse_r, out_r), 1), torch.cat((parse_r, batch["image"]), 1)), 0))
        fake_r = [[t[:n] for t in p] for p in pred_r]
        real_r = [[t[n:] for t in p] for p in pred_r]
        gan_r = float(crit(fake_r, True, for_discriminator=False))
        feat_r = float(sum(F.l1_loss(fake_r[i][j], real_r[i][j]) * 10.0 / 2 for i in range(2) for j in range(len(fake_r[i]) - 1)))
        vgg_cpu = networks.Vgg19()
        vgg_cpu.load_state_dict(vgg_cpu_sd)
        fx, fy = vgg_cpu(out_r), vgg_cpu(batch["image"])
        vl_r = float(sum(wt * F.l1_loss(a, b) for wt, a, b in zip([1.0 / 32, 1.0 / 16, 1.0 / 8, 1.0 / 4, 1.0], fx, fy)))
    print("STEP2LOSS parse agreement %.4f  image mean|d| %.3e  warped-cloth (occlusion composite) max|d| %.3e" %
          (float((parse.cpu() == parse_r).float().mean()), float((out.cpu() - out_r).abs().mean()), float((g_in.cpu()[:, 6:] - g_in_r[:, 6:]).abs().max())))
    assert float((g_in.cpu()[:, 6:] - g_in_r[:, 6:]).abs().mean()) < 2e-3  # fused warp + remove_overlap + white composite vs the torch chain
    print("STEP2LOSS gan %.4f vs %.4f | feat %.4f vs %.4f | vgg %.4f vs %.4f" % (gan, gan_r, feat, feat_r, vl, vl_r))
    assert float((parse.cpu() == parse_r).float().mean()) > 0.99  # argmax of blurred logits: a few pixels may flip under bf16
    assert abs(gan - gan_r) < 0.05 + 0.05 * abs(gan_r)
    assert abs(feat - feat_r) < 0.05 * abs(feat_r) + 0.02
    assert abs(vl - vl_r) < 0.05 * abs(vl_r) + 0.01


def test_vgg_loss_gradient_with_fused_relu_backward():
    """VGGLoss through the kernels: the ReLU backward of every Vgg19 convolution is fused into its consumers (data-gradient epilogue of the
    next convolution, max-pool backward, L1 backward — hrv_conv_params.res_mode) instead of running as a pass of its own.  Loss and
    d loss / d image vs torch autograd through the same network in fp32 on the CPU; bound = what torch's own bf16 autocast costs."""
    import networks
    from hrviton_b200 import autograd_g
    os.environ["HRV_VGG_RANDOM_INIT"] = "1"
    torch.manual_seed(3)
    vgg = networks.Vgg19().eval()
    n, h, w = 2, 128, 96
    x = (synth.uniform((n, 3, h, w), 5, "vggx")).requires_grad_(True)
    y = synth.uniform((n, 3, h, w), 5, "vggy")
    wts = [1.0 / 32, 1.0 / 16, 1.0 / 8, 1.0 / 4, 1.0]

    def ref_loss(xx, autocast):
        with torch.autocast("cpu", dtype=torch.bfloat16, enabled=autocast):
            fx, fy = vgg(xx), vgg(y)
            return sum(wt * torch.nn.functional.l1_loss(a.float(), b.float().detach()) for wt, a, b in zip(wts, fx, fy))

    l_ref = ref_loss(x, False)
    (g_ref,) = torch.autograd.grad(l_ref, x)
    l_ac = ref_loss(x, True)
    (g_ac,) = torch.autograd.grad(l_ac, x)
    vg = networks.Vgg19().eval()
    vg.load_state_dict(vgg.state_dict())
    vg = vg.cuda()
    xd = x.detach().cuda().requires_grad_(True)
    loss = autograd_g.vgg_loss(vg, wts, xd, y.cuda())
    loss.backward()
    torch.cuda.synchronize()
    g = xd.grad.cpu()
    rel = float((g - g_ref).norm() / g_ref.norm())
    rel_ac = float((g_ac - g_ref).norm() / g_ref.norm())
    print("VGGGRAD loss %.5f vs %.5f (autocast %.5f) | d/dx rel L2 %.3e (torch bf16 autocast %.3e)" % (float(loss), float(l_ref), float(l_ac), rel, rel_ac))
    assert abs(float(loss) - float(l_ref)) <= 1.25 * abs(float(l_ac) - float(l_ref)) + 2e-3 * abs(float(l_ref))
    assert rel <= 1.25 * rel_ac + 1e-2
