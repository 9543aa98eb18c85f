"""Whole-row tiles (option 37, default on): on 32- and 64-pixel-wide maps the trunk's 3x3 convs (dense-block kernel, RDB conv5,
trunk_conv) tile whole image rows from x = 0 instead of 16- or 32-pixel windows with halo columns.  The edge taps that the zero-filled
halo columns used to contribute are an explicit +0, and where a 64-pixel row spans two epilogue warps the two boundary taps are
swapped through shared memory, in the same summation order - so the outputs must be bit-identical to the tiling with halo columns.
Other widths keep the old tiling."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _with_options(opts, fn):
    from climsr_b200._lib import lib
    defaults = {37: 1, 31: 2, 25: 1}
    try:
        for k, v in opts.items():
            lib.csr_set_option(k, v)
        return fn()
    finally:
        for k in opts:
            lib.csr_set_option(k, defaults[k])


def _forward(sd, x, elev, mask, in_ch, nb):
    from climsr_b200.models import ESRGANGenerator
    net = ESRGANGenerator(in_ch, 1, 64, nb, 16)
    net.load_state_dict(sd)
    net = net.cuda().eval()
    with torch.no_grad():
        a = net(x.cuda(), elev.cuda(), mask.cuda())
        b = net(x.cuda(), elev.cuda(), mask.cuda())       # second call: CUDA-graph replay where the plan uses one
    assert torch.equal(a, b)
    return a.cpu()


@pytest.mark.parametrize("n,in_ch,h,w,nb", [
    (3, 4, 64, 64, 2),        # 64-pixel rows: two epilogue warps per row, conv5 with one shared staging buffer
    (1, 3, 37, 64, 2),        # ragged last window
    (3, 3, 64, 32, 2),        # 32-pixel rows: one warp per row
    (1, 4, 37, 32, 2),
    (2, 4, 40, 48, 2),        # 48 pixels wide: keeps the tiling with halo columns
    (64, 4, 64, 64, 11),      # cfg2
])
def test_whole_row_forward_is_bit_identical(n, in_ch, h, w, nb):
    from oracle import synth
    sd = synth.make_state_dict(in_ch, 1, 64, nb, 16, seed=41, gain=1.4)
    x, elev, mask = synth.make_inputs(n, in_ch, h, w, seed=42)
    # option 31 = 0: the dense-block kernel also runs for blocks with fewer than two windows per SM
    on = _with_options({37: 1, 31: 0}, lambda: _forward(sd, x, elev, mask, in_ch, nb))
    off = _with_options({37: 0, 31: 0}, lambda: _forward(sd, x, elev, mask, in_ch, nb))
    assert torch.isfinite(on).all()
    assert torch.equal(on, off)
    if w == 48:
        from oracle import generator as og
        want = og.generator_forward(sd, x, elev, mask)
        assert float((on - want).abs().max()) <= 1e-2


def test_whole_row_training_step_is_bit_identical():
    """cfg3 shape (16 x 32 x 32 LR, nb = 11): the training plan's forward and backward.  The output must be bit-identical.  The
    parameter gradients are not bit-reproducible even between two runs with the same tiling (fp32 partial sums land in a
    different order: ~1e-7 relative on a B200), so they are held to 1e-4 of their largest magnitude - a wrong edge tap in a
    forward or input-gradient conv moves them by orders of magnitude more."""
    from climsr_b200.models import ESRGANGenerator
    from oracle import synth
    in_ch, nb, n, h, w = 4, 11, 16, 32, 32
    sd = synth.make_state_dict(in_ch, 1, 64, nb, 16, seed=43, gain=1.2)
    x, elev, mask = synth.make_inputs(n, in_ch, h, w, seed=44)
    hr = torch.rand((n, 1, 4 * h, 4 * w), generator=torch.Generator().manual_seed(45)) * 2 - 1

    def step():
        net = ESRGANGenerator(in_ch, 1, 64, nb, 16)
        net.load_state_dict(sd)
        net = net.cuda().train()
        sr = net(x.cuda(), elev.cuda(), mask.cuda())
        F.l1_loss(sr, hr.cuda()).backward()
        return sr.detach().cpu(), {k: p.grad.detach().cpu() for k, p in net.named_parameters()}

    sr_on, g_on = _with_options({37: 1, 25: 0}, step)
    sr_off, g_off = _with_options({37: 0, 25: 0}, step)
    assert torch.equal(sr_on, sr_off)
    for k in g_off:
        assert torch.isfinite(g_on[k]).all(), k
        err = float((g_on[k] - g_off[k]).abs().max()) / max(float(g_off[k].abs().max()), 1e-30)
        assert err <= 1e-4, (k, err)
