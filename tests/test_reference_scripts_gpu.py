"""The reference's OWN training loops, unmodified, on this repository's drop-in modules.

`train_generator.train()` and `train_condition.train()` are imported from the original HR-VITON modules that build() compiles into
oracle/_ref (or a checkout named by $HRV_REFERENCE_DIR) through hrv_env (repo root first on sys.path: `networks`,
`network_generator`, `sync_batchnorm` bind to the drop-ins; shims/ supplies torchgeometry / tensorboardX / apex / numpy aliases)
and run for two iterations on a synthetic loader with the README's flags.  This is the "scripts drop in unchanged" claim of the
boundary, exercised end to end: train-mode dispatch of ConditionGenerator / tocg-D / SPADEGenerator / gen-D forward, autograd
through every kernel, the scripts' own torch glue, Adam.  Skipped where no reference checkout exists."""
import io
import contextlib
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import hrv_env  # noqa: E402

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(hrv_env.reference_dir() is None, reason="no original HR-VITON modules: build with a checkout, or set HRV_REFERENCE_DIR")]


class _Loader:
    """next_batch() of cp_dataset.CPDataLoader (cp_dataset.py:404-426) over one synthetic VITON-HD-shaped batch."""

    def __init__(self, n, h, w):
        from hrviton_b200 import train_step
        b = train_step.synthetic_batch_stage1(n, h, w, "cpu", seed=3)
        self.batch = {"agnostic": b["agnostic"], "parse": b["parse"], "densepose": b["densepose"], "parse_cloth": b["parse_cloth"],
                      "parse_agnostic": b["parse_agnostic"], "pcm": b["pcm"], "cloth_mask": {"paired": b["cloth_mask"], "unpaired": b["cloth_mask"]},
                      "cloth": {"paired": b["cloth"], "unpaired": b["cloth"]}, "image": b["image"], "pose": b["densepose"],
                      "parse_onehot": b["parse_onehot"]}  # (N,1,H,W) class ids, as cp_dataset.py:228 provides them

    def next_batch(self):
        return self.batch


class _Lpips:
    def eval(self):
        return self


def _opt(mod, argv):
    old = sys.argv
    sys.argv = ["script"] + argv
    try:
        return mod.get_opt()
    finally:
        sys.argv = old


def test_train_generator_loop_unchanged():
    import network_generator
    import networks
    tg = hrv_env.load_reference_script("train_generator")
    assert tg.SPADEGenerator is network_generator.SPADEGenerator and tg.ConditionGenerator is networks.ConditionGenerator
    h, w = 512, 384
    opt = _opt(tg, ["--name", "t", "--cuda", "True", "--gpu_ids", "0", "-b", "1", "--fine_height", str(h), "--fine_width", str(w), "--keep_step", "2",
                    "--decay_step", "0", "--display_count", "1000", "--save_count", "1000", "--tensorboard_count", "1000",
                    "--lpips_count", "1000", "--occlusion"])
    torch.manual_seed(0)
    tocg = networks.ConditionGenerator(opt, input1_nc=4, input2_nc=opt.semantic_nc + 3, output_nc=13, ngf=96, norm_layer=torch.nn.BatchNorm2d)
    generator = network_generator.SPADEGenerator(opt, 9)
    generator.cuda()
    generator.init_weights(opt.init_type, opt.init_variance)
    with contextlib.redirect_stdout(io.StringIO()):
        discriminator = tg.create_network(network_generator.MultiscaleDiscriminator, opt)  # the reference's utils.create_network
    g0 = generator.up_3.conv_0.weight_orig.detach().clone()
    d0 = discriminator.discriminator_0.model0[0].weight.detach().clone()
    u0 = generator.up_3.conv_0.weight_u.detach().clone()
    with contextlib.redirect_stdout(io.StringIO()):
        tg.train(opt, _Loader(1, h, w), None, None, tg.SummaryWriter(log_dir="unused"), tocg, generator, discriminator, _Lpips())
    torch.cuda.synchronize()
    gm = generator.module if hasattr(generator, "module") else generator
    dm = discriminator.module if hasattr(discriminator, "module") else discriminator
    assert float((gm.up_3.conv_0.weight_orig.detach() - g0).abs().max()) > 0      # Adam(G) moved the generator
    assert float((dm.discriminator_0.model0[0].weight.detach() - d0).abs().max()) > 0  # Adam(D) moved the discriminator
    assert not torch.equal(gm.up_3.conv_0.weight_u, u0)                            # train-mode spectral norm ran its power iteration
    assert all(bool(torch.isfinite(p).all()) for p in gm.parameters())


def test_train_condition_loop_unchanged():
    import networks
    tc = hrv_env.load_reference_script("train_condition")
    assert tc.ConditionGenerator is networks.ConditionGenerator and tc.define_D is networks.define_D
    opt = _opt(tc, ["--name", "t", "--gpu_ids", "0", "-b", "2", "--keep_step", "2", "--display_count", "1000", "--save_count", "1000",
                    "--tensorboard_count", "1000", "--val_count", "1000", "--cuda", "True", "--Ddownx2", "--Ddropout", "--lasttvonly",
                    "--interflowloss", "--occlusion", "--no_test_visualize"])
    torch.manual_seed(0)
    tocg = networks.ConditionGenerator(opt, input1_nc=4, input2_nc=opt.semantic_nc + 3, output_nc=opt.output_nc, ngf=96, norm_layer=torch.nn.BatchNorm2d)
    with contextlib.redirect_stdout(io.StringIO()):
        D = networks.define_D(input_nc=4 + opt.semantic_nc + 3 + opt.output_nc, Ddownx2=opt.Ddownx2, Ddropout=opt.Ddropout, n_layers_D=3,
                              spectral=opt.spectral, num_D=opt.num_D)
    w0 = tocg.flow_conv[4].weight.detach().clone()
    d0 = D.layer0[0].weight.detach().clone()
    rm0 = tocg.ClothEncoder[0].block[1].running_mean.detach().clone()
    with contextlib.redirect_stdout(io.StringIO()):
        tc.train(opt, _Loader(2, 256, 192), None, None, tc.SummaryWriter(log_dir="unused"), tocg, D)
    torch.cuda.synchronize()
    assert float((tocg.flow_conv[4].weight.detach().cpu() - w0).abs().max()) > 0
    assert float((D.layer0[0].weight.detach().cpu() - d0).abs().max()) > 0
    assert not torch.equal(tocg.ClothEncoder[0].block[1].running_mean.detach().cpu(), rm0)  # train-mode BatchNorm tracked statistics
    assert int(tocg.ClothEncoder[0].block[1].num_batches_tracked) == 2
    assert all(bool(torch.isfinite(p).all()) for p in tocg.parameters())
