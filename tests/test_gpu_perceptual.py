"""VGG19 perceptual loss (climsr_b200.losses.PerceptualLoss) and its kernels: hi/lo bf16 input conversion, the hi/lo
split-store conv epilogue (CSR_OUT_BF16_SPLIT), the 2x2 max pool over hi/lo pairs, and the loss against the float64
oracle (oracle/perceptual.py) - at the GAN step's batch, at the sizes where a plain bf16 path fails (sr close to hr), and
through SuperResolutionTask.

CPU tests: parameter layout against torchvision, state-dict loading, the oracle against torchvision, CPU inputs rejected."""
import math

import pytest
import torch
import torch.nn.functional as F

gpu = pytest.mark.gpu

# (cin, cout, hw) of the 16 convs of vgg19.features[:35] as executed at 128^2 (cin is the real input channel count)
VGG_SHAPES = [(3, 64, 128), (64, 64, 128), (64, 128, 64), (128, 128, 64), (128, 256, 32), (256, 256, 32), (256, 512, 16),
              (512, 512, 16), (512, 512, 8)]


def _smooth(n, h, w, seed):
    """A smooth field in [-1, 1] (sum of a few random low-frequency waves): hr of the accuracy tests."""
    g = torch.Generator().manual_seed(seed)
    yy = torch.linspace(0, 1, h).view(1, 1, h, 1)
    xx = torch.linspace(0, 1, w).view(1, 1, 1, w)
    f = torch.zeros((n, 1, h, w))
    for _ in range(6):
        fy, fx, ph = (torch.rand((n, 1, 1, 1), generator=g) * 6 for _ in range(3))
        f = f + torch.sin(2 * math.pi * (fy * yy + fx * xx) + ph)
    return (f / f.abs().amax(dim=(1, 2, 3), keepdim=True)).float()


def _pair_sr(hr, sigma, seed):
    g = torch.Generator().manual_seed(seed)
    return hr + sigma * torch.randn(hr.shape, generator=g)


def _split(v):
    hi = v.bfloat16()
    lo = (v - hi.float()).bfloat16()
    return hi, lo


# ------------------------------------------------------------------------------------------------ CPU
def test_parameters_match_torchvision_vgg19_features():
    tv = pytest.importorskip("torchvision")
    from climsr_b200.losses import PerceptualLoss
    ref = tv.models.vgg19(weights=None).features[:35]
    mine = PerceptualLoss().features
    a = [(k, tuple(v.shape)) for k, v in ref.state_dict().items()]
    b = [(k, tuple(v.shape)) for k, v in mine.state_dict().items()]
    assert a == b
    assert [type(m) for m in ref] == [type(m) for m in mine]
    assert not any(p.requires_grad for p in PerceptualLoss().parameters())


def test_full_vgg19_state_dict_loads_from_dict_and_path(tmp_path):
    tv = pytest.importorskip("torchvision")
    from climsr_b200.losses import PerceptualLoss
    torch.manual_seed(3)
    full = tv.models.vgg19(weights=None).state_dict()          # features.* and classifier.*
    path = tmp_path / "vgg19.pth"
    torch.save(full, path)
    for src in (full, str(path)):
        m = PerceptualLoss(src)
        for k, v in m.state_dict().items():
            assert torch.equal(v, full[k]), k
        assert not any(p.requires_grad for p in m.parameters())
    # the seeded default is reproducible and differs per seed
    assert torch.equal(PerceptualLoss(seed=4).features[0].weight, PerceptualLoss(seed=4).features[0].weight)
    assert not torch.equal(PerceptualLoss(seed=4).features[0].weight, PerceptualLoss(seed=5).features[0].weight)


def test_oracle_matches_torchvision_features_and_l1():
    tv = pytest.importorskip("torchvision")
    from climsr_b200.losses import PerceptualLoss
    from oracle import perceptual as op
    sd = PerceptualLoss(seed=1).state_dict()
    net = tv.models.vgg19(weights=None).features[:35]
    net.load_state_dict({k[len("features."):]: v for k, v in sd.items()})
    net = net.double().eval()
    hr = _smooth(2, 32, 40, 0)
    sr = _pair_sr(hr, 0.05, 1)
    with torch.no_grad():
        want = F.l1_loss(net(hr.double().repeat(1, 3, 1, 1)), net(sr.double().repeat(1, 3, 1, 1)))
        got = op.perceptual_loss(sd, hr, sr)
        want3 = F.l1_loss(net(hr.double().repeat(1, 3, 1, 1) * 0.5), net(sr.double().repeat(1, 3, 1, 1)))
        got3 = op.perceptual_loss(sd, hr.repeat(1, 3, 1, 1) * 0.5, sr.repeat(1, 3, 1, 1))
    assert got.dtype == torch.float64
    assert abs(float(got - want)) <= 1e-10 * max(1.0, float(want))
    assert abs(float(got3 - want3)) <= 1e-10 * max(1.0, float(want3))


def test_cpu_inputs_raise_csr_error():
    from climsr_b200 import CsrError
    from climsr_b200.losses import PerceptualLoss
    m = PerceptualLoss()
    x = torch.rand(1, 1, 16, 16)
    with pytest.raises(CsrError):
        m(x, x)


def test_shapes_rejected_before_any_device_work():
    from climsr_b200.losses import PerceptualLoss
    m = PerceptualLoss()
    for a, b in ((torch.rand(1, 2, 32, 32), torch.rand(1, 2, 32, 32)),      # channels
                 (torch.rand(1, 1, 15, 32), torch.rand(1, 1, 15, 32)),      # H < 16
                 (torch.rand(1, 1, 32, 32), torch.rand(1, 1, 32, 16)),      # mismatch
                 (torch.rand(1, 32, 32), torch.rand(1, 32, 32))):           # not 4-D
        with pytest.raises(ValueError):
            m(a, b)


# ------------------------------------------------------------------------------------------------ GPU: kernels
@gpu
@pytest.mark.parametrize("c", [1, 3])
def test_split_conversion(c):
    from climsr_b200 import ops
    g = torch.Generator().manual_seed(c)
    x = torch.rand((3, c, 37, 50), generator=g) * 2 - 1
    out = ops.nchw_to_nhwc_split(x.cuda(), 16).cpu()
    xt = x.permute(0, 2, 3, 1)
    hi, lo = out[..., :c], out[..., c:2 * c]
    assert torch.equal(hi.view(torch.int16), xt.bfloat16().view(torch.int16))
    rec = hi.float() + lo.float()
    assert float(((rec - xt).abs() - 2.0 ** -16 * xt.abs()).max()) <= 0
    assert not out[..., 2 * c:].float().any()


def _conv_case(cin, cout, hw, n=32):
    """The split-store conv of one VGG layer at batch n over a hi/lo input, against float64."""
    from climsr_b200 import ops
    g = torch.Generator().manual_seed(cin * 7 + cout + hw)
    dev = "cuda"
    if cin <= 3:
        x = (torch.rand((n, cin, hw, hw), generator=g) * 2 - 1).to(dev)
        inp = ops.nchw_to_nhwc_split(x, 16)
        cin_exec = 2 * cin
        hi, lo = inp[..., :cin].float(), inp[..., cin:2 * cin].float()
    else:
        v = torch.relu(torch.randn((n, hw, hw, cin), generator=g)).to(dev)       # post-ReLU activations of the previous layer
        hi, lo = _split(v)
        inp = torch.cat([hi, lo], -1).contiguous()
        hi, lo = hi.float(), lo.float()
        cin_exec = 2 * cin
    w = (torch.randn((cout, cin, 3, 3), generator=g) * (2.0 / (cout * 9)) ** 0.5).to(dev)
    b = (torch.rand((cout,), generator=g) * 0.2 - 0.1).to(dev)
    wx = torch.cat([w, w], 1)
    assert wx.shape[1] == cin_exec
    out = ops.conv2d_nhwc(inp, wx, b, act="relu", out_mode="split")
    assert out.shape == (n, hw, hw, 2 * cout)
    xr = (hi.double() + lo.double()).permute(0, 3, 1, 2)                       # the reconstructed input
    wb = w.bfloat16().double()                                                 # the kernel's weights are bf16
    want = torch.relu(F.conv2d(xr, wb, b.double(), padding=1)).permute(0, 2, 3, 1)
    mag = (F.conv2d(xr.abs(), wb.abs(), b.double().abs(), padding=1)).permute(0, 2, 3, 1)
    ohi, olo = out[..., :cout].float(), out[..., cout:].float()
    got = ohi.double() + olo.double()
    # fp32 accumulation of K = 9 * cin_exec products, and the pair's own representation error (2^-17 relative)
    err = (got - want).abs() - 2.0 ** -16 * mag
    assert float(err.max()) <= 0, float(((got - want).abs() / mag.clamp_min(1e-30)).max())
    # |lo| is at most half a bf16 ulp of hi (and 0 where hi is 0)
    m, e = torch.frexp(ohi)
    half_ulp = torch.ldexp(torch.ones_like(ohi), e - 9)
    assert bool((olo.abs() <= half_ulp).all())
    assert bool((olo[ohi == 0] == 0).all())
    # every output-channel part of gridDim.y wrote its hi and its lo range
    assert bool(torch.isfinite(got).all())
    for k in range(0, cout, 64):
        assert bool((ohi[..., k:k + 64] != 0).any()) and bool((olo[..., k:k + 64] != 0).any())


@gpu
@pytest.mark.parametrize("cin,cout,hw", VGG_SHAPES)
def test_split_store_conv_every_vgg_layer_shape(cin, cout, hw):
    _conv_case(cin, cout, hw)


@gpu
def test_split_store_conv_gray_input():
    _conv_case(1, 64, 128)                 # cin' = 2 at 128^2: conv1_1 of a 1-channel input


@gpu
@pytest.mark.parametrize("hw", [128, 64, 32, 16, 113])
def test_maxpool_split_bit_exact(hw):
    from climsr_b200 import ops
    c = 64
    g = torch.Generator().manual_seed(hw)
    v = torch.randn((3, hw, hw + 2, c), generator=g)
    v[0, 5, 7, 3] = float("nan")
    v[2, hw - 1, 0, 60] = float("nan")
    hi, lo = _split(v)
    got = ops.maxpool2x2_split(torch.cat([hi, lo], -1).cuda()).cpu()
    rec = (hi.float() + lo.float()).permute(0, 3, 1, 2).cuda()
    pooled = F.max_pool2d(rec, 2).permute(0, 2, 3, 1).cpu()
    whi, wlo = _split(pooled)
    assert got.shape == (3, hw // 2, (hw + 2) // 2, 2 * c)
    for a, b in ((got[..., :c], whi), (got[..., c:], wlo)):
        na, nb = torch.isnan(a.float()), torch.isnan(b.float())
        assert torch.equal(na, nb)
        assert torch.equal(a.view(torch.int16)[~na], b.view(torch.int16)[~nb])
    assert bool(torch.isnan(got[0, 2, 3, 3].float()))


@gpu
def test_maxpool_split_rejects_bad_shapes():
    from climsr_b200 import CsrError, ops
    with pytest.raises(CsrError):
        ops.maxpool2x2_split(torch.zeros((1, 1, 8, 32), dtype=torch.bfloat16, device="cuda"))     # h < 2
    with pytest.raises(CsrError):
        ops.maxpool2x2_split(torch.zeros((1, 8, 8, 24), dtype=torch.bfloat16, device="cuda"))     # c = 12


# ------------------------------------------------------------------------------------------------ GPU: the loss
def _oracle(sd, hr, sr, emulate="none"):
    from oracle import perceptual as op
    with torch.no_grad():
        return float(op.perceptual_loss({k: v.cuda() for k, v in sd.items()}, hr.cuda(), sr.cuda(), emulate))


@gpu
@pytest.mark.parametrize("sigma", [0.05, 0.01, 0.002])
def test_loss_matches_float64_oracle(sigma):
    """At sigma = 0.002 a plain bf16 path is ~100 % off (oracle emulate="bf16"): this is the test that pins the hi/lo design."""
    from climsr_b200.losses import PerceptualLoss
    m = PerceptualLoss(seed=0).cuda()
    hr = _smooth(16, 128, 128, 1)
    sr = _pair_sr(hr, sigma, 2)
    got = m(hr.cuda(), sr.cuda())
    assert got.shape == () and got.dtype == torch.float32 and not got.requires_grad
    want = _oracle(m.state_dict(), hr, sr)
    rel = abs(float(got) - want) / want
    print(f"sigma {sigma}: loss {float(got):.6e} oracle {want:.6e} rel {rel:.2e}")
    assert rel <= 1e-2


@gpu
def test_loss_at_europe_hr_size():
    from climsr_b200.losses import PerceptualLoss
    m = PerceptualLoss(seed=2).cuda()
    hr = _smooth(2, 452, 452, 3)
    sr = _pair_sr(hr, 0.01, 4)
    got = float(m(hr.cuda(), sr.cuda()))
    want = _oracle(m.state_dict(), hr, sr)
    assert abs(got - want) / want <= 1e-2, (got, want)


@gpu
def test_reference_self_test_zero_and_positive():
    from climsr_b200.losses import PerceptualLoss
    m = PerceptualLoss().cuda()
    g = torch.Generator().manual_seed(9)
    x = (torch.rand((3, 1, 64, 80), generator=g) * 2 - 1).cuda()
    y = (torch.rand((3, 1, 64, 80), generator=g) * 2 - 1).cuda()
    assert float(m(x, x)) == 0.0
    assert float(m(x, y)) > 0


@gpu
def test_gray_input_equals_repeated_three_channels():
    from climsr_b200.losses import PerceptualLoss
    m = PerceptualLoss(seed=3).cuda()
    hr = _smooth(4, 96, 64, 5).cuda()
    sr = _pair_sr(hr.cpu(), 0.01, 6).cuda()
    a = float(m(hr, sr))
    b = float(m(hr.repeat(1, 3, 1, 1), sr.repeat(1, 3, 1, 1)))
    assert abs(a - b) <= 1e-2 * b, (a, b)


@gpu
def test_no_gradient_reaches_sr():
    from climsr_b200 import losses
    m = losses.PerceptualLoss().cuda()
    hr = _smooth(2, 64, 64, 7).cuda()
    sr0 = _pair_sr(hr.cpu(), 0.05, 8).cuda()
    sr = sr0.clone().requires_grad_(True)
    (0.01 * losses.l1_loss(sr, hr) + m(hr, sr)).backward()
    g1 = sr.grad.clone()
    sr2 = sr0.clone().requires_grad_(True)
    (0.01 * losses.l1_loss(sr2, hr)).backward()
    assert torch.equal(g1, sr2.grad)
    assert not m(hr, sr).requires_grad


@gpu
def test_load_state_dict_repacks():
    from climsr_b200.losses import PerceptualLoss
    m = PerceptualLoss(seed=0).cuda()
    hr = _smooth(2, 64, 64, 10)
    sr = _pair_sr(hr, 0.05, 11)
    before = float(m(hr.cuda(), sr.cuda()))
    m.load_state_dict(PerceptualLoss(seed=7).state_dict())
    after = float(m(hr.cuda(), sr.cuda()))
    want = _oracle(m.state_dict(), hr, sr)
    assert after != before
    assert abs(after - want) / want <= 1e-2, (after, want)


@gpu
def test_gan_task_logs_the_perceptual_term():
    from climsr_b200.losses import PerceptualLoss
    from climsr_b200.models import ESRGANGenerator
    from climsr_b200.models.discriminator import Discriminator
    from climsr_b200.task import SuperResolutionTask
    torch.manual_seed(0)
    perc = PerceptualLoss(seed=0).cuda()
    task = SuperResolutionTask(ESRGANGenerator(4, 1, 64, 1, 16).cuda(), discriminator=Discriminator().cuda(),
                               perceptual_criterion=perc).train()
    g = torch.Generator().manual_seed(5)
    n = 2
    mask = (torch.rand((n, 1, 128, 128), generator=g) > 0.3).float()
    batch = {"lr": (torch.rand((n, 4, 32, 32), generator=g) * 2 - 1).cuda(), "hr": (torch.rand((n, 1, 128, 128), generator=g) * 2 - 1).cuda(),
             "elevation": (torch.rand((n, 1, 128, 128), generator=g) * mask).cuda(), "mask": mask.cuda(),
             "original_data": (torch.rand((n, 1, 128, 128), generator=g) * 40 - 10).cuda(),
             "min": torch.tensor([-30.0, -25.0], dtype=torch.float64).cuda(), "max": torch.tensor([35.0, 40.0], dtype=torch.float64).cuda()}
    for p in task.discriminator.parameters():
        p.requires_grad_(False)
    out = task.training_step(batch, 0, optimizer_idx=0)
    log = out["log"]
    with torch.no_grad():
        _, sr = task.common_step(batch)
        standalone = float(perc(batch["hr"], sr))
    p = float(log["train/perceptual_loss"])
    assert p > 0 and abs(p - standalone) <= 1e-5 * standalone, (p, standalone)
    want = 0.01 * float(log["train/pixel_level_loss"].detach()) + 1.0 * p + 0.005 * float(log["train/adversarial_loss"].detach())
    assert abs(float(out["loss"].detach()) - want) <= 1e-5 * abs(want)
    out["loss"].backward()
    assert all(q.grad is not None for q in task.generator.parameters())
    task.eval()
    val = task.validation_step(batch)
    assert float(val["val/perceptual_loss"]) > 0
