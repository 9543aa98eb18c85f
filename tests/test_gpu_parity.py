"""GPU parity tests proper: the CUDA path through the C-ABI vs the oracle / golden vectors of the reference.

Tolerances (BASELINE.json north_star): generator max-abs error <= 1e-2 in normalised units (bf16 I/O, fp32
accumulate); PSNR within 0.01 dB; SSIM within 1e-4; integer-count metrics (RegressionAccuracy) exact.
"""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

GEN_TOL = 1e-2


def _bf(t):
    return t.to(torch.bfloat16).float()


def _ref_conv(x, w, b, act, slope=0.0):
    y = F.conv2d(_bf(x).double(), _bf(w).double(), b.double(), padding=(w.shape[2] // 2, w.shape[3] // 2))
    if act == "lrelu":
        y = F.leaky_relu(y, 0.2)
    elif act == "lrelu_slope":
        y = F.leaky_relu(y, slope)
    elif act == "relu":
        y = F.relu(y)
    return y.float()


def _nhwc(x, c):
    return F.pad(x.permute(0, 2, 3, 1), (0, c - x.shape[1])).to(torch.bfloat16).contiguous().cuda()


CONV_CASES = [
    # n, h, w, cin, cout, k, act, in_c       (the layer shapes of esrgan.py / srcnn.py plus ragged / empty-ish edges)
    (1, 8, 14, 16, 16, 1, "none", 64),
    (2, 16, 16, 64, 16, 3, "lrelu", 128),      # RDB conv1
    (2, 16, 16, 80, 16, 3, "lrelu", 128),      # RDB conv2
    (1, 16, 16, 112, 16, 3, "lrelu", 128),     # RDB conv4
    (2, 16, 16, 128, 64, 3, "none", 128),      # RDB conv5 (gc=16)
    (1, 24, 24, 192, 64, 3, "none", 192),      # RDB conv5 (gc=32): cout split over two launches
    (1, 33, 45, 64, 64, 3, "lrelu", 64),       # ragged edges, several tiles
    (1, 1, 1, 64, 64, 3, "none", 64),          # single pixel
    (3, 5, 130, 64, 64, 3, "none", 64),        # wide, short
    (1, 20, 40, 4, 64, 3, "none", 64),         # conv_first, cin 4 -> 16
    (1, 20, 40, 2, 64, 3, "none", 64),         # conv_first, cin 2 (reference's own test case)
    (1, 40, 40, 64, 1, 3, "none", 64),         # conv_last (ragged cout)
    (1, 40, 40, 3, 64, 9, "relu", 64),         # srcnn.conv1
    (1, 40, 40, 64, 32, 1, "relu", 64),        # srcnn.conv2
    (1, 40, 40, 32, 1, 5, "none", 64),         # srcnn.conv3
    (1, 113, 113, 64, 64, 3, "lrelu", 64),     # Europe-extent LR raster
    (2, 9, 11, 64, 24, 3, "relu", 64),         # cout multiple of 8 but not 16
    (1, 7, 33, 64, 20, 3, "none", 64),         # ragged cout: per-element store path
    # the discriminator's ten convs at the GAN step's batch 16, as the same-convs over their padded maps it runs
    # ("lrelu_slope=s": LeakyReLU(s) epilogue; stride 2 reads every second pixel of the same-conv's output)
    (16, 130, 130, 1, 64, 3, "lrelu_slope=0.01", 64),      # stage 1 conv_a: one input channel in a 64-channel buffer
    (16, 130, 130, 64, 64, 3, "lrelu_slope=0.01", 64),     # stage 1 conv_b (stride 2)
    (16, 66, 66, 64, 128, 3, "lrelu_slope=0.01", 64),      # stage 2 conv_a
    (16, 66, 66, 128, 128, 3, "lrelu_slope=0.01", 128),    # stage 2 conv_b
    (16, 34, 34, 128, 256, 3, "lrelu_slope=0.01", 128),    # stage 3 conv_a
    (16, 34, 34, 256, 256, 3, "lrelu_slope=0.01", 256),    # stage 3 conv_b: k-block weight streaming, output-channel parts
    (16, 18, 18, 256, 512, 3, "lrelu_slope=0.01", 256),    # stage 4 conv_a
    (16, 18, 18, 512, 512, 3, "lrelu_slope=0.01", 512),    # stage 4 conv_b
    (16, 8, 8, 512, 512, 3, "lrelu_slope=0.2", 512),       # conv4 (valid)
    (16, 6, 6, 512, 512, 3, "none", 512),                  # conv5 (valid)
]


@pytest.mark.parametrize("n,h,w,cin,cout,k,act,in_c", CONV_CASES)
def test_conv_matches_fp32_reference(n, h, w, cin, cout, k, act, in_c):
    from climsr_b200 import ops
    act, _, slope = act.partition("=")
    slope = float(slope or 0.0)
    g = torch.Generator().manual_seed(n * 1000 + h * 10 + cin + k)
    x = torch.rand((n, cin, h, w), generator=g) * 2 - 1
    wt = (torch.rand((cout, cin, k, k), generator=g) * 2 - 1) / (cin * k * k) ** 0.5
    b = torch.rand((cout,), generator=g) - 0.5
    xin = _nhwc(x, in_c)
    if cin % 16 == 0 and in_c > cin:
        xin[..., cin:] = 9.0          # channels beyond cin must never be multiplied
    out = ops.conv2d_nhwc(xin, wt.cuda(), b.cuda(), act=act, act_slope=slope)
    got = out[..., :cout].float().cpu().permute(0, 3, 1, 2)
    # fp64 on the GPU for the large layers (the same fp64 arithmetic, seconds instead of minutes on the host)
    dev = "cuda" if n * h * w * cin * cout > 1 << 26 else "cpu"
    want = _ref_conv(x.to(dev), wt.to(dev), b.to(dev), act, slope).cpu()
    assert torch.isfinite(got).all()
    # bf16 output rounding: half an ulp relative (2^-9) plus fp32 accumulation noise
    assert float((got - want).abs().max()) <= 2.0 ** -8 * max(1.0, float(want.abs().max()))


def test_conv_epilogue_variants():
    from climsr_b200 import ops
    g = torch.Generator().manual_seed(5)
    n, h, w = 2, 12, 20
    x = torch.rand((n, 64, h, w), generator=g) * 2 - 1
    wt = (torch.rand((64, 64, 3, 3), generator=g) * 2 - 1) / 24
    b = torch.rand((64,), generator=g) - 0.5
    r1 = torch.rand((n, 64, h, w), generator=g) * 2 - 1
    r2 = torch.rand((n, 64, h, w), generator=g) * 2 - 1
    y = _ref_conv(x, wt, b, "none")
    # x5*0.2 + x, then *0.2 + x_rrdb (esrgan.py:38,54)
    out = ops.conv2d_nhwc(_nhwc(x, 64), wt.cuda(), b.cuda(), res1=_nhwc(r1, 64), scale1=0.2, res2=_nhwc(r2, 64), scale2=0.2)
    want = (y * 0.2 + _bf(r1)) * 0.2 + _bf(r2)
    assert float((out.float().cpu().permute(0, 3, 1, 2) - want).abs().max()) <= 2.0 ** -7
    # in-place residual: out aliases res2 (RDB3 writes the RRDB output over the RRDB input)
    buf = _nhwc(r2, 64)
    ops.conv2d_nhwc(_nhwc(x, 64), wt.cuda(), b.cuda(), out=buf, res1=_nhwc(r1, 64), scale1=0.2, res2=buf, scale2=0.2)
    assert float((buf.float().cpu().permute(0, 3, 1, 2) - want).abs().max()) <= 2.0 ** -7
    # nearest x2 then conv + lrelu (esrgan.py:94,97): executed as four 2x2 sub-pixel convs with summed weights
    out = ops.conv2d_nhwc(_nhwc(x, 64), wt.cuda(), b.cuda(), act="lrelu", in_up2=True)
    up = F.interpolate(_bf(x), scale_factor=2, mode="nearest")
    want = F.leaky_relu(F.conv2d(up.double(), wt.double(), b.double(), padding=1), 0.2).float()
    assert out.shape == (n, 2 * h, 2 * w, 64)
    # phase weights are sums of up to four bf16-rounded-after-summing taps: compare against fp32 weights, bf16 tolerance
    assert float((out.float().cpu().permute(0, 3, 1, 2) - want).abs().max()) <= 2.0 ** -6
    # fp32 planar (final layer)
    w1 = (torch.rand((1, 64, 5, 5), generator=g) * 2 - 1) / 40
    b1 = torch.rand((1,), generator=g)
    out = ops.conv2d_nhwc(_nhwc(x, 64), w1.cuda(), b1.cuda(), out_mode="f32_planar")
    assert float((out.cpu() - _ref_conv(x, w1, b1, "none")).abs().max()) <= 1e-4
    # write-into-concat-slice (torch.cat of esrgan.py:34-37 without the copy)
    cat = torch.zeros((n, h, w, 128), dtype=torch.bfloat16).cuda()
    cat[..., :64] = _nhwc(x, 64)
    w16 = (torch.rand((16, 64, 3, 3), generator=g) * 2 - 1) / 24
    b16 = torch.rand((16,), generator=g) - 0.5
    ops.conv2d_nhwc(cat, w16.cuda(), b16.cuda(), act="lrelu", out=cat, out_coff=64)
    got = cat[..., 64:80].float().cpu().permute(0, 3, 1, 2)
    assert float((got - _ref_conv(x, w16, b16, "lrelu")).abs().max()) <= 2.0 ** -7
    assert bool((cat[..., 80:] == 0).all()) and bool((cat[..., :64] == _nhwc(x, 64)).all())
    # per-element store path (option 4) must agree bit-for-bit with the TMA-store path
    # (hybrid tap fold off: it only exists for staged stores and adds the last tap inside the accumulator - another summation order)
    from climsr_b200._lib import lib
    lib.csr_set_option(35, 0)
    try:
        a = ops.conv2d_nhwc(_nhwc(x, 64), wt.cuda(), b.cuda(), act="lrelu")
        lib.csr_set_option(4, 1)
        c = ops.conv2d_nhwc(_nhwc(x, 64), wt.cuda(), b.cuda(), act="lrelu")
    finally:
        lib.csr_set_option(4, 0)
        lib.csr_set_option(35, 1)
    assert torch.equal(a, c)


@pytest.mark.parametrize("n,h,w,cin,cout,k,in_c,in_coff", [
    (2, 5, 33, 64, 16, 3, 128, 0),      # second M tile of the window mostly below the image
    (1, 12, 61, 112, 16, 3, 128, 0),    # one and a half windows, two k-blocks
    (3, 24, 24, 16, 16, 3, 128, 64),    # 16 input channels at an offset: 32-byte window rows
    (1, 17, 40, 32, 32, 3, 64, 0),      # 32 input channels: 64-byte rows; N = 96 -> four accumulators
    (1, 40, 40, 64, 32, 1, 64, 0),      # 1x1 (srcnn.conv2 shape)
    (1, 21, 19, 32, 1, 5, 64, 0),       # srcnn.conv3 shape -> bf16 path here (fp32 planar is covered by the generator tests)
])
def test_thin_layer_variants_are_bit_identical(n, h, w, cin, cout, k, in_c, in_coff):
    """Two-tile windows (option 18), eight accumulator buffers (19) and narrow window boxes (17) only change how tiles are
    scheduled and how many bytes are moved: every combination must give the SAME bits as the plain kernel, and those must
    match the fp32 reference conv."""
    from climsr_b200 import ops
    from climsr_b200._lib import lib
    g = torch.Generator().manual_seed(100 + h + w)
    x = torch.rand((n, in_c, h, w), generator=g) * 2 - 1
    wt = (torch.rand((cout, cin, k, k), generator=g) * 2 - 1) / (3 * k * cin ** 0.5)
    b = torch.rand((cout,), generator=g) - 0.5
    xin = _nhwc(x, in_c)
    outs = []
    try:
        for tall, acc8, narrow in ((0, 0, 0), (1, 0, 0), (1, 1, 0), (1, 1, 1), (0, 0, 1)):
            lib.csr_set_option(18, tall)
            lib.csr_set_option(19, acc8)
            lib.csr_set_option(17, narrow)
            outs.append(ops.conv2d_nhwc(xin, wt.cuda(), b.cuda(), act="lrelu", in_coff=in_coff))
    finally:
        for key in (17, 18, 19):
            lib.csr_set_option(key, 1)
    for o in outs[1:]:
        assert torch.equal(o, outs[0])
    want = _ref_conv(x[:, in_coff:in_coff + cin], wt, b, "lrelu")
    got = outs[0][..., :cout].float().cpu().permute(0, 3, 1, 2)
    assert float((got - want).abs().max()) <= 2.0 ** -7 * max(1.0, float(want.abs().max()))


def test_conv_transposed_and_gate():
    """Input-gradient conv (transposed/flipped weights) with in-place accumulate and LeakyReLU-derivative gate: the building
    block of the dense-block backward (autograd of esrgan.py:33-38)."""
    from climsr_b200 import ops
    g = torch.Generator().manual_seed(11)
    n, h, w = 2, 13, 21
    cin_f, cout_f = 80, 16                       # forward conv2 of an RDB: 80 -> 16
    wt = (torch.rand((cout_f, cin_f, 3, 3), generator=g) * 2 - 1) / 20
    gy = torch.rand((n, cout_f, h, w), generator=g) * 2 - 1
    acc0 = torch.rand((n, cin_f, h, w), generator=g) * 2 - 1          # gradient already accumulated in the buffer
    fwd = torch.rand((n, cin_f, h, w), generator=g) * 2 - 1           # saved forward activations (sign -> lrelu')
    want = F.conv_transpose2d(_bf(gy).double(), _bf(wt).double(), padding=1).float() + _bf(acc0)
    gate = torch.where(_bf(fwd) > 0, 1.0, 0.2)
    gate[:, :64] = 1.0
    want = want * gate
    gbuf = torch.zeros((n, h, w, 128), dtype=torch.bfloat16).cuda()
    gbuf[..., :cin_f] = acc0.permute(0, 2, 3, 1).to(torch.bfloat16).cuda()
    gbuf[..., 80:96] = gy.permute(0, 2, 3, 1).to(torch.bfloat16).cuda()
    fbuf = torch.zeros((n, h, w, 128), dtype=torch.bfloat16).cuda()
    fbuf[..., :cin_f] = fwd.permute(0, 2, 3, 1).to(torch.bfloat16).cuda()
    ops.conv2d_nhwc(gbuf, wt.cuda(), None, in_coff=80, transposed=True, out=gbuf, out_coff=0, res1=gbuf, scale1=1.0,
                    gate=fbuf, gate_from=64)
    got = gbuf[..., :cin_f].float().cpu().permute(0, 3, 1, 2)
    assert float((got - want).abs().max()) <= 2.0 ** -7 * max(1.0, float(want.abs().max()))
    assert torch.equal(gbuf[..., 80:96].cpu(), gy.permute(0, 2, 3, 1).to(torch.bfloat16))


def _run_generator(sd, x, elev, mask, in_ch, nb, gc):
    from climsr_b200.models import ESRGANGenerator
    net = ESRGANGenerator(in_ch, 1, 64, nb, gc)
    net.load_state_dict(sd)
    net = net.cuda().eval()
    with torch.no_grad():
        return net(x.cuda(), elev.cuda(), mask.cuda()).cpu()


def test_generator_matches_reference_golden_refinit(golden_dir):
    """Weights, inputs and output all produced by the UNMODIFIED reference module (oracle/make_golden.py)."""
    z = np.load(os.path.join(golden_dir, "gen_tiny_refinit.npz"))
    sd = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd/")}
    got = _run_generator(sd, torch.from_numpy(z["x"]), torch.from_numpy(z["elev"]), torch.from_numpy(z["mask"]), 2, 1, 16)
    assert got.shape == z["sr"].shape
    assert np.abs(got.numpy() - z["sr"]).max() <= GEN_TOL


@pytest.mark.parametrize("name", ["gen_hydra_seeded.npz", "gen_default_seeded.npz"])
def test_generator_matches_reference_golden_seeded(golden_dir, name):
    from oracle import synth
    z = np.load(os.path.join(golden_dir, name))
    in_ch, nb, gc, n, h, w = (int(v) for v in z["meta"])
    x, elev, mask = synth.make_inputs(n, in_ch, h, w, seed=1)
    gains = [float(g) for g in z["gains"]]
    for tag, gain in zip(("sr", "sr_trained", "sr_stress"), gains):
        sd = synth.make_state_dict(in_ch, 1, 64, nb, gc, seed=0, gain=gain)
        got = _run_generator(sd, x, elev, mask, in_ch, nb, gc).numpy()
        err = np.abs(got - z[tag]).max()
        if tag == "sr_stress":
            # chaotic gain: any bf16-I/O implementation (the reference under bf16 included) is accurate to ~2 % of range
            assert err <= 0.025 * np.abs(z[tag]).max(), (tag, err)
        else:
            assert err <= GEN_TOL, (tag, err)


def _fulldepth_case(golden_dir, name):
    from oracle import synth
    z = np.load(os.path.join(golden_dir, "gen_fulldepth.npz"))
    in_ch, nb, gc, n, h, w, wseed, iseed = (int(v) for v in z[name + "_meta"])
    sd = synth.make_state_dict(in_ch, 1, 64, nb, gc, seed=wseed, gain=float(z[name + "_gain"]))
    x, elev, mask = synth.make_inputs(n, in_ch, h, w, seed=iseed, blocky_mask=name.startswith("cfg4"))
    return sd, x, elev, mask, (in_ch, nb, gc), torch.from_numpy(z[name])


@pytest.mark.parametrize("name", ["cfg2_default", "cfg2_trained", "cfg4_trained", "default64_trained"])
def test_generator_matches_reference_golden_fulldepth(golden_dir, name):
    """FULL-depth outputs of the unmodified reference module at the BASELINE configs' own tile sizes: two cfg2 tiles (4x64x64 LR,
    nb=11, gc=16: multi-window rows, two-tile windows, 33 in-place concat rotations), the cfg4 Europe raster (3x113x113: ragged
    last windows) and a class-default (nb=23, gc=32) 64x64 tile, at default and "trained-like" weight gains."""
    sd, x, elev, mask, (in_ch, nb, gc), want = _fulldepth_case(golden_dir, name)
    got = _run_generator(sd, x, elev, mask, in_ch, nb, gc)
    assert got.shape == want.shape
    err = float((got - want).abs().max())
    assert err <= GEN_TOL, (name, err)


def test_cfg5_chain_generator_then_masked_metrics_matches_reference_sr(golden_dir):
    """BASELINE cfg5 end to end: the masked validation metrics of the CUDA generator's output (CUDA metric kernels) against the
    same metrics of the REFERENCE module's output (oracle metric restatement, float64) for the same hr / original / mask:
    PSNR within 0.01 dB, SSIM within 1e-4 (north_star), the remaining means within 1e-3 relative."""
    from climsr_b200._lib import METRIC_KEYS
    from climsr_b200.metrics import masked_val_metrics_raw
    from oracle import metrics as om
    from oracle import synth
    sd, x, elev, mask, (in_ch, nb, gc), sr_ref = _fulldepth_case(golden_dir, "cfg4_trained")
    t = synth.make_targets(sr_ref, seed=4)
    mn, mx = t["min"].double(), t["max"].double()
    orig = om.denormalized_original(t["hr"].double(), mn, mx).float()
    want = om.val_test_step(sr_ref, t["hr"], orig, mask, mn, mx, loss="l1")
    from climsr_b200.models import ESRGANGenerator
    net = ESRGANGenerator(in_ch, 1, 64, nb, gc)
    net.load_state_dict(sd)
    net = net.cuda().eval()
    with torch.no_grad():
        sr = net(x.cuda(), elev.cuda(), mask.cuda())
        got = masked_val_metrics_raw(sr, t["hr"].cuda(), orig.cuda(), mask.cuda(), mn.cuda(), mx.cuda()).cpu()
    v = {k: float(got[i]) for i, k in enumerate(METRIC_KEYS)}
    assert 20.0 < float(want["psnr"]) < 50.0                      # a realistic operating point, not a degenerate one
    assert abs(v["psnr"] - float(want["psnr"])) <= 0.01
    assert abs(v["ssim"] - float(want["ssim"])) <= 1e-4
    for k in ("mae", "mse", "rmse", "mape", "smape", "r2"):
        assert abs(v[k] - float(want[k])) <= 3e-3 * max(1.0, abs(float(want[k]))), k      # 0.01 dB of PSNR = 0.23 % of the MSE
    assert abs(v["l1_loss"] - float(want["loss"])) <= 1e-3 * max(1e-3, float(want["loss"]))


@pytest.mark.parametrize("n,in_ch,h,w", [(1, 3, 113, 113), (16, 4, 32, 32), (3, 4, 20, 36), (1, 1, 9, 7)])
def test_generator_matches_oracle_shapes(n, in_ch, h, w):
    """cfg4 (Europe extent 113x113, in=3), cfg1 (16x32x32, in=4), ragged and tiny rasters vs the oracle (Hydra cfg, nb cut to 2
    so the CPU oracle stays in seconds; full depth is covered by the golden tests)."""
    from oracle import generator as og
    from oracle import synth
    nb, gc = 2, 16
    sd = synth.make_state_dict(in_ch, 1, 64, nb, gc, seed=2)
    x, elev, mask = synth.make_inputs(n, in_ch, h, w, seed=3)
    with torch.no_grad():
        want = og.generator_forward(sd, x, elev, mask)
    got = _run_generator(sd, x, elev, mask, in_ch, nb, gc)
    assert got.shape == want.shape == (n, 1, 4 * h, 4 * w)
    assert float((got - want).abs().max()) <= GEN_TOL


def test_reference_shape_test_case():
    """tests/models/test_esrgan.py:7-22 of the reference, verbatim shapes (in=2, batch 32, 32x32 -> 128x128)."""
    from climsr_b200.models import ESRGANGenerator
    model = ESRGANGenerator(2, 1).cuda()
    x = torch.rand((32, 2, 32, 32)).cuda()
    elev = torch.rand((32, 1, 128, 128)).cuda()
    mask = torch.rand((32, 1, 128, 128)).cuda()
    with torch.no_grad():
        out = model.forward(x, elev, mask)
    assert out.shape == (32, 1, 128, 128)
    assert torch.isfinite(out).all()


def test_generator_properties_at_full_size():
    """BASELINE cfg2 size (64 x 64x64 LR): size-independent properties instead of a CPU oracle run.
    (1) batch independence: tile i of the batch == the same tile run alone, bit-exact;
    (2) determinism: two runs are bit-identical; (3) repacking after an in-place weight update changes the output."""
    from climsr_b200.models import ESRGANGenerator
    torch.manual_seed(0)
    net = ESRGANGenerator(4, 1, 64, 11, 16).cuda().eval()
    g = torch.Generator().manual_seed(1)
    x = (torch.rand((64, 4, 64, 64), generator=g) * 2 - 1).cuda()
    elev = (torch.rand((64, 1, 256, 256), generator=g) * 2 - 1).cuda()
    mask = (torch.rand((64, 1, 256, 256), generator=g) > 0.3).float().cuda()
    with torch.no_grad():
        a = net(x, elev, mask)
        b = net(x, elev, mask)
        assert torch.equal(a, b)
        for i in (0, 37, 63):
            single = net(x[i:i + 1], elev[i:i + 1], mask[i:i + 1])
            assert torch.equal(single[0], a[i])
        net.conv_last.bias.add_(1.0)
        c = net(x, elev, mask)
    assert not torch.equal(a, c)
    assert torch.isfinite(c).all()


def test_regression_accuracy_kats_through_cabi():
    """The nine known-answer cases of tests/metrics/test_regresion_accuracy.py:12-108, routed through csr_masked_metrics
    (z-score scaler with mean 0 / std 1 and an all-land mask make the kernel's denormalised pair equal (preds, targets))."""
    from climsr_b200._lib import METRIC_KEYS
    from climsr_b200.metrics import masked_val_metrics_raw
    shape = (3, 1, 128, 128)
    eps_idx = {0.1: METRIC_KEYS.index("acc@0.1"), 0.25: METRIC_KEYS.index("acc@0.25"), 1.0: METRIC_KEYS.index("acc@1")}
    ones = torch.ones(shape)
    for eps, idx in eps_idx.items():
        g = torch.Generator().manual_seed(int(eps * 100))
        cases = [(torch.zeros(shape), ones + (1 if eps == 1.0 else 0), 0.0), (ones.clone(), ones, 1.0),
                 (ones - torch.rand(shape, generator=g) / 100, ones, 1.0)]
        for preds, targets, expected in cases:
            v = masked_val_metrics_raw(preds.cuda(), targets.cuda(), targets.cuda(), ones.cuda(), zscore=(0.0, 1.0)).cpu()
            assert float(v[idx]) == expected


@pytest.mark.parametrize("n,H,W,blocky", [(2, 64, 64, False), (3, 45, 50, True), (1, 452, 452, True), (4, 128, 128, False)])
def test_masked_metrics_match_oracle(n, H, W, blocky):
    from climsr_b200._lib import METRIC_KEYS
    from climsr_b200.metrics import masked_val_metrics, masked_val_metrics_raw
    from oracle import metrics as om
    from oracle import synth
    g = torch.Generator().manual_seed(n + H)
    sr = (torch.rand(n, 1, H, W, generator=g) * 2 - 1) * 0.8
    t = synth.make_targets(sr, seed=4)
    if blocky:
        low = torch.rand((n, 1, max(H // 16, 1), max(W // 16, 1)), generator=g)
        mask = (F.interpolate(low, size=(H, W), mode="nearest") > 0.3).float()
    else:
        mask = (torch.rand(n, 1, H, W, generator=g) > 0.3).float()
    # batch["min"] / batch["max"] are float64 (N,) tensors in the reference; "original" is the float32 raster of the dataset
    mn, mx = t["min"].double() + 0.1234567891234, t["max"].double() - 0.9876543219876
    orig = om.denormalized_original(t["hr"].double(), mn, mx).float()
    want = om.val_test_step(sr, t["hr"], orig, mask, mn, mx, loss="l1")
    want_mse = om.val_test_step(sr, t["hr"], orig, mask, mn, mx, loss="mse")["loss"]
    got = masked_val_metrics_raw(sr.cuda(), t["hr"].cuda(), orig.cuda(), mask.cuda(), mn.cuda(), mx.cuda()).cpu()
    for i, k in enumerate(METRIC_KEYS):
        ref = float(want["loss"]) if k == "l1_loss" else float(want_mse) if k == "mse_loss" else float(want[k])
        if k.startswith("acc@"):
            # integer counts: EXACT (the kernel denormalises in float64 with the reference's operation order and a true division)
            assert round(float(got[i]) * n * H * W) == round(ref * n * H * W), k
            assert float(got[i]) == float(torch.tensor(ref, dtype=torch.float64).float()), k
        elif k == "psnr":
            assert abs(float(got[i]) - ref) <= 0.01, k
        elif k == "ssim":
            assert abs(float(got[i]) - ref) <= 1e-4, k
        else:
            assert abs(float(got[i]) - ref) <= 1e-4 * max(1.0, abs(ref)), k
    d = masked_val_metrics(sr.cuda(), t["hr"].cuda(), orig.cuda(), mask.cuda(), t["min"].cuda(), t["max"].cuda(), prefix="test")
    assert "test/acc@01.25" in d and "test/loss" in d and len(d) == 18     # the reference's key typo is kept (task.py:325)


def test_masked_metrics_zscore_and_mask_invariance():
    from climsr_b200.metrics import masked_val_metrics_raw
    from oracle import metrics as om
    g = torch.Generator().manual_seed(9)
    n, H, W = 2, 40, 36
    sr = torch.rand(n, 1, H, W, generator=g) * 2 - 1
    hr = (sr + 0.05 * torch.randn(sr.shape, generator=g))
    mask = (torch.rand(n, 1, H, W, generator=g) > 0.4).float()
    orig = hr * 8.5 + 12.0
    want = om.val_test_step(sr, hr, orig, mask, zscore=(12.0, 8.5))
    a = masked_val_metrics_raw(sr.cuda(), hr.cuda(), orig.cuda(), mask.cuda(), zscore=(12.0, 8.5)).cpu()
    assert abs(float(a[10]) - float(want["mae"])) <= 1e-4 * max(1.0, float(want["mae"]))
    sr2 = sr.clone()
    sr2[~mask.bool()] += 100.0     # ocean pixels never contribute (task.py:288-291)
    b = masked_val_metrics_raw(sr2.cuda(), hr.cuda(), orig.cuda(), mask.cuda(), zscore=(12.0, 8.5)).cpu()
    assert torch.equal(a, b)


@pytest.mark.parametrize("shape", [(2, 1, 64, 64), (3, 1, 45, 51), (1, 1, 1, 3), (4, 1, 256, 256)])
def test_pixel_losses_value_and_gradient(shape):
    """csr_l1_loss / csr_mse_loss (core/task.py:141): value and d loss / d sr vs torch, ragged numel, exact zeros (sign(0) = 0)."""
    from climsr_b200 import losses
    g = torch.Generator().manual_seed(sum(shape))
    sr = (torch.rand(shape, generator=g) * 2 - 1)
    hr = (torch.rand(shape, generator=g) * 2 - 1)
    hr.view(-1)[::7] = sr.view(-1)[::7]
    for ours, ref in ((losses.l1_loss, F.l1_loss), (losses.mse_loss, F.mse_loss)):
        a = sr.clone().cuda().requires_grad_(True)
        b = sr.clone().double().requires_grad_(True)
        lo = ours(a, hr.cuda())
        lr = ref(b, hr.double())
        (lo * 3.0).backward()
        (lr * 3.0).backward()
        assert abs(float(lo.detach()) - float(lr.detach())) <= 1e-6 * max(1.0, abs(float(lr.detach())))
        assert float((a.grad.cpu().double() - b.grad).abs().max()) <= 1e-6 * float(b.grad.abs().max() + 1e-30) + 1e-12
    with torch.no_grad():
        assert losses.l1_loss(sr.cuda(), hr.cuda()).requires_grad is False


def test_tiled_inference_matches_untiled():
    """cfg4: Europe-extent raster (113x113 LR, in=3) as 8 halo-padded row bands (one per GPU of a box) vs the un-tiled run."""
    from climsr_b200.models import ESRGANGenerator
    from climsr_b200.tiling import band_plan, tiled_forward_all
    from oracle import synth
    torch.manual_seed(0)
    net = ESRGANGenerator(3, 1, 64, 11, 16).cuda().eval()
    x, elev, mask = (t.cuda() for t in synth.make_inputs(1, 3, 113, 113, seed=1))
    with torch.no_grad():
        full = net(x, elev, mask)
        tiled = tiled_forward_all(net, x, elev, mask, bands=8, halo=16)
        rough = tiled_forward_all(net, x, elev, mask, bands=8, halo=0)
    assert tiled.shape == full.shape == (1, 1, 452, 452)
    assert len(band_plan(113, 8, 16)) == 8
    e16, e0 = float((tiled - full).abs().max()), float((rough - full).abs().max())
    assert e16 <= 2e-3 and e0 > 10 * e16 + 1e-3, (e16, e0)


def test_host_pipeline_matches_direct_calls():
    """HostPipeline (pinned host -> device -> host, copies overlapped with compute) returns exactly what direct forward calls do,
    in submission order."""
    from climsr_b200.models import ESRGANGenerator
    from climsr_b200.pipeline import HostPipeline
    torch.manual_seed(0)
    net = ESRGANGenerator(3, 1, 64, 1, 16).cuda().eval()
    g = torch.Generator().manual_seed(4)
    batches = []
    for _ in range(5):
        x = (torch.rand((2, 3, 12, 16), generator=g) * 2 - 1).pin_memory()
        e = torch.rand((2, 1, 48, 64), generator=g).pin_memory()
        m = (torch.rand((2, 1, 48, 64), generator=g) > 0.3).float().pin_memory()
        batches.append((x, e, m))
    pipe = HostPipeline(net, (2, 3, 12, 16), depth=2)
    got = []
    for b in batches:
        r = pipe.submit(*b)
        if r is not None:
            got.append(r.clone())
    got += [t.clone() for t in pipe.drain()]
    assert len(got) == 5
    with torch.no_grad():
        for (x, e, m), o in zip(batches, got):
            assert torch.equal(net(x.cuda(), e.cuda(), m.cuda()).cpu(), o)


def test_minmax_scaler_kernels_match_reference_golden(golden_dir):
    """csr_minmax_normalize / csr_minmax_denormalize_mask against the reference's MinMaxScaler outputs (bit-exact: float64
    arithmetic, one rounding) - normalization.py:37-84, inference.py:73-76."""
    from climsr_b200.normalization import MinMaxScaler
    g = np.load(os.path.join(golden_dir, "normalization.npz"))
    sc = MinMaxScaler(feature_range=(-1.0, 1.0))
    raw = torch.from_numpy(g["raw"]).cuda()
    h, w = raw.shape[1:]
    elev_lr = torch.rand((h, w)) * 2 - 1
    mask_lr = (torch.rand((h, w)) > 0.3).float()
    x = sc.normalize(raw, g["mins"], g["maxes"], [elev_lr, mask_lr]).cpu()
    assert x.shape == (raw.shape[0], 3, h, w)
    assert np.array_equal(x[:, 0].numpy(), g["norm"])
    assert torch.equal(x[:, 1], elev_lr.expand(raw.shape[0], h, w)) and torch.equal(x[:, 2], mask_lr.expand(raw.shape[0], h, w))
    assert np.array_equal(MinMaxScaler().normalize(raw[:1], g["mins"][:1], g["maxes"][:1]).cpu().numpy()[0, 0], g["norm01"])
    sr = torch.from_numpy(g["sr"]).cuda()
    mask = torch.from_numpy(g["mask"].astype(np.float32)).cuda()
    post = sc.denormalize(sr, g["mins"], g["maxes"], mask).cpu().numpy()
    assert np.array_equal(post, g["post"], equal_nan=True)
    post_n = sc.denormalize(sr, g["mins"], g["maxes"], mask.expand(sr.shape[0], 1, -1, -1).contiguous()).cpu().numpy()
    assert np.array_equal(post_n, g["post"], equal_nan=True)
    with pytest.raises(ValueError):
        sc.normalize(raw, g["mins"][:2], g["maxes"])


def test_raster_pipeline_matches_oracle_chain():
    """Raw LR rasters -> normalise -> generator -> denormalise -> NaN mask, all on device with overlapped copies
    (RasterPipeline), against the oracle chain (oracle.normalization + oracle.generator) - inference.py:56-82."""
    from climsr_b200.models import ESRGANGenerator
    from climsr_b200.pipeline import RasterPipeline
    from oracle import generator as og
    from oracle import normalization as on
    from oracle import synth
    n, h, w = 2, 12, 20
    sd = synth.make_state_dict(3, 1, 64, 1, 16, seed=9)
    net = ESRGANGenerator(3, 1, 64, 1, 16)
    net.load_state_dict(sd)
    net = net.cuda().eval()
    rng = np.random.default_rng(4)
    mask = (rng.uniform(size=(1, 1, 4 * h, 4 * w)) > 0.3).astype(np.float32)
    elev = (rng.uniform(-1, 1, size=(1, 1, 4 * h, 4 * w)).astype(np.float32)) * mask
    elev_lr, mask_lr = elev[0, 0, ::4, ::4].copy(), mask[0, 0, ::4, ::4].copy()
    pipe = RasterPipeline(net, n, h, w, torch.from_numpy(elev), torch.from_numpy(mask), torch.from_numpy(elev_lr), torch.from_numpy(mask_lr))
    batches, outs = [], []
    for b in range(3):
        raw = rng.uniform(-30, 40, size=(n, h, w)).astype(np.float32)
        raw[np.broadcast_to(mask_lr == 0, raw.shape)] = np.nan
        mins = np.array([-45.5 - b, -50.25], dtype=np.float64)
        maxes = np.array([44.0, 47.5 + b], dtype=np.float64)
        batches.append((raw, mins, maxes))
        r = pipe.submit(torch.from_numpy(raw).pin_memory(), torch.from_numpy(mins).pin_memory(), torch.from_numpy(maxes).pin_memory())
        if r is not None:
            outs.append(r.clone())
    outs += [o.clone() for o in pipe.drain()]
    assert len(outs) == 3
    for (raw, mins, maxes), got in zip(batches, outs):
        x = on.lr_input(raw, mins, maxes, elev_lr, mask_lr)
        e = np.broadcast_to(elev, (n, 1, 4 * h, 4 * w)).copy()
        m = np.broadcast_to(mask, (n, 1, 4 * h, 4 * w)).copy()
        sr = og.generator_forward(sd, torch.from_numpy(x), torch.from_numpy(e), torch.from_numpy(m)).numpy()
        want = on.postprocess(sr, mask, mins, maxes)
        got = got.numpy()
        assert np.array_equal(np.isnan(got), np.isnan(want))
        land = ~np.isnan(want)
        # 1e-2 in normalised units (bf16 path) = 1e-2 * (max - min) / 2 in physical units
        tol = 1e-2 * (maxes - mins).max() / 2
        assert np.abs(got[land] - want[land]).max() <= tol


def test_lr_input_kernel_matches_numpy_cv2_golden(golden_dir):
    """csr_lr_input_from_hr against numpy flips / rot90 + cv2 INTER_NEAREST resize (climate_dataset.py:98-172): all 16
    augmentation codes, bit-exact; un-augmented non-square rasters; a full-size batch against the oracle."""
    from climsr_b200.data import aug_code, make_lr_batch, random_aug_codes
    from oracle import lr_input as ol
    g = np.load(os.path.join(golden_dir, "lr_input.npz"))
    hr, elev, mask = (torch.from_numpy(g[k]).cuda() for k in ("hr", "elev", "mask"))
    x, hr2, el2, mk2 = make_lr_batch(hr, elev, mask, torch.from_numpy(g["codes"]))
    assert np.array_equal(x.cpu().numpy(), g["x"])
    assert np.array_equal(hr2.cpu().numpy(), g["hr_aug"]) and np.array_equal(el2.cpu().numpy(), g["elev_aug"])
    assert np.array_equal(mk2.cpu().numpy(), g["mask_aug"])
    assert aug_code(True, False, 3) == 13
    # no augmentation, non-square raster
    r = torch.from_numpy(g["rect"])[None, None].cuda()
    x0, a0, _, _ = make_lr_batch(r, r * 0.5, (r > 0).float())
    assert np.array_equal(x0[0, 0].cpu().numpy(), g["rect_lr"]) and torch.equal(x0[0, 1], x0[0, 0] * 0.5) and a0.data_ptr() == r.data_ptr()
    with pytest.raises(ValueError):
        make_lr_batch(r, r, r, torch.tensor([4]))             # rot90 by 1 on a 20x36 raster
    # training-size batch (cfg3: 16 x 128x128) with drawn codes, against the oracle
    gen = torch.Generator().manual_seed(8)
    n, S = 16, 128
    hr = torch.rand((n, 1, S, S), generator=gen) * 2 - 1
    elev = torch.rand((n, 1, S, S), generator=gen) * 2 - 1
    mask = (torch.rand((n, 1, S, S), generator=gen) > 0.3).float()
    codes = random_aug_codes(n, gen)
    assert int(codes.max()) <= 15 and len(set(codes.tolist())) > 4
    got = make_lr_batch(hr.cuda(), elev.cuda(), mask.cuda(), codes)
    want = ol.training_batch(hr.numpy(), elev.numpy(), mask.numpy(), codes.numpy())
    for a, b in zip(got, want):
        assert np.array_equal(a.cpu().numpy(), b)


@pytest.mark.parametrize("n,in_ch,h,w,nb", [(4, 4, 64, 64, 3), (1, 3, 113, 113, 2), (3, 4, 20, 36, 2), (1, 1, 9, 7, 1), (16, 4, 32, 32, 2), (150, 4, 16, 16, 1)])
def test_dense_block_kernel_is_bit_identical_to_per_layer_launches(n, in_ch, h, w, nb):
    """conv1..conv4 of every dense block as ONE persistent launch with tile-level dependencies (rdb_tc.cu, option 27, default)
    against four per-layer launches: same tiles, same MMA order, same epilogue arithmetic -> bit-identical outputs.  Shapes:
    cfg2 tiles (several windows per CTA), the Europe raster (ragged last windows), a ragged small raster, a raster smaller than
    one window, cfg1, and more windows than SMs with a single window row per image."""
    from climsr_b200._lib import lib
    from climsr_b200.models import ESRGANGenerator
    from oracle import synth
    sd = synth.make_state_dict(in_ch, 1, 64, nb, 16, seed=6, gain=1.4)
    x, elev, mask = synth.make_inputs(n, in_ch, h, w, seed=7)
    outs = []
    try:
        lib.csr_set_option(31, 0)                                 # also for blocks below the default two-windows-per-SM threshold
        for dense in (1, 0, 1):
            lib.csr_set_option(27, dense)
            net = ESRGANGenerator(in_ch, 1, 64, nb, 16)
            net.load_state_dict(sd)
            net = net.cuda().eval()
            with torch.no_grad():
                a = net(x.cuda(), elev.cuda(), mask.cuda())
                b = net(x.cuda(), elev.cuda(), mask.cuda())          # second call: CUDA-graph replay where the plan uses one
            assert torch.equal(a, b)
            outs.append(a.cpu())
            del net
    finally:
        lib.csr_set_option(27, 1)
        lib.csr_set_option(31, 2)
    assert torch.equal(outs[0], outs[1])
    assert torch.equal(outs[0], outs[2])


@pytest.mark.parametrize("n,in_ch,h,w", [(2, 4, 64, 64), (1, 3, 113, 113), (3, 4, 20, 36), (1, 1, 9, 7)])
def test_hybrid_tap_fold_matches_full_fold(n, in_ch, h, w):
    """Option 35 (default 1): in the epilogue-bound 64-channel early-release layers (HRconv, the upconv phases) the LAST horizontal tap
    is an MMA of its own over an A operand shifted by one pixel (descriptor start + 128 bytes inside the 128B-swizzled window) that
    accumulates into the previous tap's columns, instead of a third column group summed by shuffles.  Same products, the last tap is
    added inside the accumulator instead of in the epilogue -> equal up to fp32 summation order and single bf16 rounding flips."""
    from climsr_b200._lib import lib
    from climsr_b200.models import ESRGANGenerator
    from oracle import synth
    sd = synth.make_state_dict(in_ch, 1, 64, 1, 16, seed=36, gain=1.2)
    x, elev, mask = synth.make_inputs(n, in_ch, h, w, seed=37)
    outs = []
    try:
        for hyb in (1, 0):
            lib.csr_set_option(35, hyb)
            net = ESRGANGenerator(in_ch, 1, 64, 1, 16)
            net.load_state_dict(sd)
            net = net.cuda().eval()
            with torch.no_grad():
                outs.append(net(x.cuda(), elev.cuda(), mask.cuda()).cpu())
            del net
    finally:
        lib.csr_set_option(35, 1)
    scale = max(1.0, float(outs[1].abs().max()))
    assert float((outs[0] - outs[1]).abs().max()) <= 3e-3 * scale, float((outs[0] - outs[1]).abs().max())


@pytest.mark.parametrize("n,in_ch,h,w", [(2, 4, 64, 64), (1, 3, 113, 113), (3, 4, 20, 36), (1, 1, 9, 7)])
def test_merged_subpixel_phase_launches_are_bit_identical(n, in_ch, h, w):
    """Option 34 (default on): the two sub-pixel phases of nearest-x2 + conv that share a kernel specialisation run as ONE launch with
    the vertical phase on gridDim.y (two launches per upconv instead of four).  Same tiles, same arithmetic -> bit-identical."""
    from climsr_b200._lib import lib
    from climsr_b200.models import ESRGANGenerator
    from oracle import synth
    sd = synth.make_state_dict(in_ch, 1, 64, 1, 16, seed=26, gain=1.2)
    x, elev, mask = synth.make_inputs(n, in_ch, h, w, seed=27)
    outs = []
    try:
        for merged in (1, 0):
            lib.csr_set_option(34, merged)
            net = ESRGANGenerator(in_ch, 1, 64, 1, 16)
            net.load_state_dict(sd)
            net = net.cuda().eval()
            with torch.no_grad():
                outs.append(net(x.cuda(), elev.cuda(), mask.cuda()).cpu())
            del net
    finally:
        lib.csr_set_option(34, 1)
    assert torch.equal(outs[0], outs[1])


@pytest.mark.parametrize("n,in_ch,h,w", [(4, 4, 64, 64), (1, 3, 113, 113), (3, 4, 20, 36), (1, 1, 9, 7), (2, 4, 5, 33)])
def test_fused_hr_tail_matches_separate_launches(n, in_ch, h, w):
    """Option 33 (inference plans; default 3 = both).  Bit 0: srcnn.conv2 (1x1, 64 -> 32, ReLU) as a second MMA over srcnn.conv1's staged
    bf16 tile (conv_tc.cu FUSE_T = 1) - same bf16 operands, same four k-steps in the same order -> BIT-IDENTICAL to the two launches.
    Bit 1: conv_last (3x3, 64 -> 1) as nine 1x1 'tap' channels computed by a second MMA inside HRconv's epilogue (FUSE_T = 2) + the
    shifted tap sum (tap_sum_kernel) - same products, another fp32 summation order, then the bf16 rounding of the SRCNN input: equal to a
    small fraction of the output scale.  In both cases the 64-channel HR map never reaches memory."""
    from climsr_b200._lib import lib
    from climsr_b200.models import ESRGANGenerator
    from oracle import synth
    sd = synth.make_state_dict(in_ch, 1, 64, 1, 16, seed=16, gain=1.2)
    x, elev, mask = synth.make_inputs(n, in_ch, h, w, seed=17)
    outs = {}
    try:
        for fuse in (1, 0, 3, 2):
            lib.csr_set_option(33, fuse)
            net = ESRGANGenerator(in_ch, 1, 64, 1, 16)
            net.load_state_dict(sd)
            net = net.cuda().eval()
            with torch.no_grad():
                a = net(x.cuda(), elev.cuda(), mask.cuda())
                b = net(x.cuda(), elev.cuda(), mask.cuda())
            assert torch.equal(a, b)
            outs[fuse] = a.cpu()
            del net
    finally:
        lib.csr_set_option(33, 3)
    assert all(torch.isfinite(o).all() for o in outs.values())
    assert torch.equal(outs[1], outs[0])
    assert torch.equal(outs[3], outs[2])
    scale = max(1.0, float(outs[0].abs().max()))
    assert float((outs[3] - outs[0]).abs().max()) <= 2e-3 * scale, float((outs[3] - outs[0]).abs().max())


@pytest.mark.parametrize("key,value", [(None, None), (33, 0), (36, 0)])
def test_plan_num_launches_matches_a_forward(key, value):
    """csr_plan_num_launches is exactly what one forward without graph replay adds to the launch counter, for the default HR tail
    (tap sum inside the SRCNN input pack), the separate tap sum (option 36 = 0) and the unfused tail (option 33 = 0); cfg4 shapes."""
    from climsr_b200 import kernel_launch_count
    from climsr_b200._lib import lib
    from climsr_b200.models import ESRGANGenerator
    from oracle import synth
    x, elev, mask = (t.cuda() for t in synth.make_inputs(1, 3, 113, 113, seed=41))
    lib.csr_set_option(11, 0)
    if key is not None:
        lib.csr_set_option(key, value)
    try:
        net = ESRGANGenerator(3, 1, 64, 11, 16).cuda().eval()
        with torch.no_grad():
            net(x, elev, mask)                       # packs the weights and creates the plan
            before = kernel_launch_count()
            net(x, elev, mask)
            launched = kernel_launch_count() - before
        assert launched == lib.csr_plan_num_launches(net._plan(1, 113, 113, x.device))
    finally:
        lib.csr_set_option(11, 1)
        if key is not None:
            lib.csr_set_option(key, {33: 3, 36: 1}[key])


@pytest.mark.parametrize("tag", ["small", "hydra"])
def test_rcan_matches_reference_golden(golden_dir, tag):
    """SURVEY 8f row 4: climsr_b200.models.rcan.RCAN (conv kernel + channel-attention / PixelShuffle kernels) against the outputs
    of the UNMODIFIED reference RCAN at a reduced depth and at the Hydra depth (10 groups x 20 blocks, conf/generator/rcan.yaml),
    default initialisation re-derived from the seed (same parameter creation order, pinned in tests/test_oracle.py)."""
    from climsr_b200 import CsrError
    from climsr_b200.models.rcan import RCAN
    from oracle import synth
    z = np.load(os.path.join(golden_dir, "rcan.npz"))
    ng, nbk, n, h, w, seed = (int(v) for v in z[tag + "_meta"])
    torch.manual_seed(seed)
    net = RCAN(n_resgroups=ng, n_resblocks=nbk, n_feats=64, reduction=16, scaling_factor=4, in_channels=3, out_channels=1).cuda().eval()
    x, elev, mask = synth.make_inputs(n, 3, h, w, seed=50 + seed)
    with torch.no_grad():
        got = net(x.cuda(), elev.cuda(), mask.cuda())
        again = net(x.cuda(), elev.cuda(), mask.cuda())           # second call: cached weight packs
    assert torch.equal(got, again)
    assert got.shape == z[tag].shape
    err = float((got.cpu() - torch.from_numpy(z[tag])).abs().max())
    assert err <= GEN_TOL, (tag, err)
    with pytest.raises(CsrError):                                 # training is not implemented for this model: loud, not silent
        net(x.cuda(), elev.cuda(), mask.cuda())
    with torch.no_grad():
        net.tail[1].bias.add_(0.25)                               # in-place update -> version bump -> repack
        moved = net(x.cuda(), elev.cuda(), mask.cuda())
    assert float((moved - got).abs().max()) > 1e-3
