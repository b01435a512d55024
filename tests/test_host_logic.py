"""CPU: host-side logic of the drop-in modules that needs no GPU — loss modules, grid, checkpoint io, init, weight packing,
tile pickers (the numerics of the kernels themselves are covered by the -m gpu tests)."""
import io
import contextlib
import os
import types

import numpy as np
import pytest
import torch

from helpers import gen_opt, tocg_opt
from hrviton_b200 import ops


def test_make_grid_matches_reference_formula():
    import networks
    g4 = networks.make_grid(2, 5, 7, types.SimpleNamespace(cuda=False))
    g3 = networks.make_grid(2, 5, 7)  # stale 3-argument form (train_condition.py:241)
    assert g4.shape == (2, 5, 7, 2)
    assert torch.equal(g4[0, 0, :, 0], torch.linspace(-1, 1, 7)) and torch.equal(g4[0, :, 0, 1], torch.linspace(-1, 1, 5))
    assert torch.equal(g3.cpu(), g4)


def test_hinge_ganloss_matches_reference_semantics():
    import network_generator
    crit = network_generator.GANLoss("hinge")
    p = [[torch.tensor([[0.5, -2.0]]), torch.tensor([[1.5, 0.2]])], [torch.tensor([[3.0]])]]  # 2 scales, last entry = logits
    # discriminator, real: -mean(min(x-1,0)) per scale, averaged over scales (network_generator.py:369-398)
    want = (-(torch.clamp(p[0][-1] - 1, max=0)).mean() + -(torch.clamp(p[1][-1] - 1, max=0)).mean()) / 2
    assert torch.allclose(crit(p, True, for_discriminator=True), want)
    want_f = (-(torch.clamp(-p[0][-1] - 1, max=0)).mean() + -(torch.clamp(-p[1][-1] - 1, max=0)).mean()) / 2
    assert torch.allclose(crit(p, False, for_discriminator=True), want_f)
    assert torch.allclose(crit(p, True, for_discriminator=False), (-(p[0][-1].mean()) - p[1][-1].mean()) / 2)
    with pytest.raises(ValueError):
        network_generator.GANLoss("bogus")


def test_lsgan_ganloss():
    import networks
    crit = networks.GANLoss(use_lsgan=True)
    pred = [[torch.tensor([[0.5, 2.0]])], [torch.tensor([[1.0]])]]
    assert torch.allclose(crit(pred, True), ((pred[0][-1] - 1) ** 2).mean() + ((pred[1][-1] - 1) ** 2).mean())
    assert torch.allclose(crit(pred, False), (pred[0][-1] ** 2).mean() + (pred[1][-1] ** 2).mean())


def test_checkpoint_roundtrip(tmp_path):
    import networks
    opt = tocg_opt(False)
    with contextlib.redirect_stdout(io.StringIO()):
        a = networks.ConditionGenerator(opt, 4, 16, 13, ngf=8, norm_layer=torch.nn.BatchNorm2d)
        b = networks.ConditionGenerator(opt, 4, 16, 13, ngf=8, norm_layer=torch.nn.BatchNorm2d)
    path = os.path.join(tmp_path, "sub", "tocg.pth")
    networks.save_checkpoint(a, path, opt)  # creates the directory like the reference (networks.py:411-417)
    networks.load_checkpoint(b, path, opt)
    for (k, v), (_, w) in zip(a.state_dict().items(), b.state_dict().items()):
        assert torch.equal(v, w), k


def test_init_weights_and_print_network(capsys):
    import network_generator
    d = network_generator.MultiscaleDiscriminator(gen_opt(256, 256))
    d.print_network()
    assert "MultiscaleDiscriminator" in capsys.readouterr().out
    d.init_weights("xavier", 0.02)
    w = d.discriminator_0.model0[0].weight
    assert float(w.std()) < 0.02  # xavier_normal with gain 0.02
    with pytest.raises(NotImplementedError):
        d.init_weights("bogus")


def test_tile_pickers():
    assert ops.pick_bk(128) == 64 and ops.pick_bk(80) == 32 and ops.pick_bk(7) == 16 and ops.pick_bk(1040) == 64
    for n in (16, 160, 256, 544, 1056, 2080, 2048):
        bn = ops.pick_bn(n)
        assert bn % 16 == 0 and 16 <= bn <= 256
        assert ops.round_up(n, bn) - n < 0.08 * n + 16  # padding stays small


def test_s2d_weight_equivalence_on_cpu():
    """The stride-2 -> space-to-depth rewrite is exact: conv(x, w, stride 2) == conv(s2d(x), s2d_weight(w), stride 1), and the
    weight gradient of the rewritten convolution maps back onto the 4x4 / 3x3 parameter."""
    import torch.nn.functional as F
    for k, pad, h, w in [(4, 2, 11, 8), (3, 1, 10, 8), (3, 1, 9, 7), (4, 2, 12, 9)]:
        x = torch.randn(2, 5, h, w)
        wt = torch.randn(6, 5, k, k, requires_grad=True)
        ref = F.conv2d(x, wt, stride=2, padding=pad)
        c8 = 8
        xp = F.pad(x, (0, w % 2, 0, h % 2, 0, c8 - 5))
        n, c, hh, ww = xp.shape
        s = xp.reshape(n, c, hh // 2, 2, ww // 2, 2).permute(0, 3, 5, 1, 2, 4).reshape(n, 4 * c, hh // 2, ww // 2)  # channel (py*2+px)*c8+ci
        got = F.conv2d(s, ops.s2d_weight(wt, pad), stride=1, padding=1)[:, :, :ref.shape[2], :ref.shape[3]]
        assert torch.allclose(got, ref, atol=1e-4), (k, pad, h, w)
        got.square().sum().backward()
        g1 = wt.grad.clone()
        wt.grad = None
        ref.square().sum().backward()
        assert float((g1 - wt.grad).abs().max()) < 1e-3 * float(wt.grad.abs().max()), (k, pad, h, w)


def test_im2col_weight_equivalence_on_cpu():
    """ops.im2col_weight: a 3x3 convolution over a few-channel map == a 1x1 convolution over the tap-major columns that
    hrv_im2col produces (column j = tap*C + ci, zero padded to 64) — checked with F.unfold as the column builder."""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 7, 9, 6, generator=g)
    w = torch.randn(12, 7, 3, 3, generator=g, requires_grad=True)
    cols = F.unfold(x, 3, padding=1).reshape(2, 7, 9, 9 * 6).permute(0, 2, 1, 3).reshape(2, 63, 9, 6)  # tap-major
    cols = F.pad(cols, (0, 0, 0, 0, 0, 1))
    wc = ops.im2col_weight(w, 64)
    assert wc.shape == (12, 64, 1, 1)
    out = F.conv2d(cols, wc)
    ref = F.conv2d(x, w, padding=1)
    assert float((out - ref).abs().max()) < 1e-5
    # the index shuffle is differentiable: the 1x1 weight gradient maps back onto the 3x3 parameter
    out.square().sum().backward()
    g1 = w.grad.clone()
    w.grad = None
    ref.square().sum().backward()
    assert float((g1 - w.grad).abs().max()) < 1e-3 * float(w.grad.abs().max())


def test_label_regrouping_table():
    """train_step.GROUP_OF_13 is the inverse of the 7-group label table (train_generator.py:261-269): every class in exactly one group."""
    from hrviton_b200 import train_step
    assert len(train_step.GROUP_OF_13) == 13
    for k, grp in enumerate(train_step.GROUP_OF_13):
        assert k in train_step.LABELS7[grp]
    assert sorted(sum(train_step.LABELS7, [])) == list(range(13))


def test_gaussian_blur_restatement_is_normalised_and_separable():
    """gaussian_blur_15_3 (the checker of the fused parse kernel): constant image -> constant away from the zero-padded border,
    and equal to the explicit 15x15 outer-product kernel."""
    import torch.nn.functional as F
    from hrviton_b200 import train_step
    x = torch.ones(1, 2, 40, 40)
    y = train_step.gaussian_blur_15_3(x)
    assert float((y[..., 10:30, 10:30] - 1).abs().max()) < 1e-5
    k = torch.arange(15, dtype=torch.float32) - 7
    g = torch.exp(-(k * k) / 18.0)
    g = g / g.sum()
    z = torch.randn(1, 1, 32, 32, generator=torch.Generator().manual_seed(1))
    ref = F.conv2d(z, torch.outer(g, g)[None, None], padding=7)
    assert float((train_step.gaussian_blur_15_3(z) - ref).abs().max()) < 1e-5


def test_gaussian_blur_restatement_matches_scipy_gaussian_filter():
    """Independent pin of the one glue op whose reference implementation (torchgeometry 0.1.2, `tgm.image.GaussianBlur((15,15),(3,3))`,
    train_generator.py:181 / test_generator.py:91) is absent from this image: its published algorithm is a normalised sampled
    Gaussian exp(-x^2 / 2 sigma^2) of 15 taps applied separably with zero padding.  scipy.ndimage.gaussian_filter with
    truncate = 7/3 (radius int(truncate*sigma + 0.5) = 7), mode='constant', cval=0 is the same filter written by someone else."""
    import numpy as np
    import scipy.ndimage as ndi
    from hrviton_b200 import train_step
    rng = np.random.default_rng(3)
    x = rng.standard_normal((2, 3, 37, 29)).astype(np.float32)
    ours = train_step.gaussian_blur_15_3(torch.from_numpy(x)).numpy()
    want = np.stack([np.stack([ndi.gaussian_filter(x[n, c].astype(np.float64), sigma=3.0, truncate=7.0 / 3.0 + 1e-9, mode="constant", cval=0.0)
                               for c in range(3)]) for n in range(2)])
    assert ours.shape == want.shape
    assert float(np.abs(ours - want).max()) < 2e-6
    # the shim the reference scripts import resolves to the same filter on CPU tensors
    import hrv_env
    hrv_env.install()
    import torchgeometry as tgm
    shim = tgm.image.GaussianBlur((15, 15), (3, 3))(torch.from_numpy(x)).numpy()
    assert float(np.abs(shim - want).max()) < 2e-6
