"""The discriminator path kernel by kernel, against float64 references, at the GAN step's batch size (16 images of 128 x 128,
DESIGN.md section 6d).

Every reference is float64 and reads the same bf16 operands the kernel reads: activations as stored, conv weights rounded to
bf16.  Inputs use the S layout of include/climsr_b200.h (discriminator section): a layer's real outputs are the logical
pixels (off + step*i, off + step*j) of its buffer.  Pixels that are not logical are filled with NaN (proves they are never
read), outputs are pre-filled with NaN (proves every element is written) and accumulating outputs (dgamma, dbeta, dW, db)
start at 1 (proves +=).

Bounds.  Glue kernels that only move or add a few bf16 values: bit-exact, or one bf16 ulp of the bf16-rounded fp64 value.
BatchNorm statistics: 1e-4 relative (fp32 per-thread partials of x - pivot); the arithmetic that follows them: 1e-5.
Convolutions: 2^-8 * max(1, max|ref|) (test_gpu_parity.py); weight gradients: 1e-3 * max|ref| (test_gpu_backward.py);
fp32 dot products: 1e-5 * (|x| . |W|^T + |b|) elementwise.

The last test is a CPU test: it chains the same fp64 per-layer references and checks that they reproduce stock PyTorch's
forward and autograd gradients of the module's own containers, which pins the references themselves.
"""
import copy
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

SLOPE, SLOPE_TAIL = 0.01, 0.2
EPS, MOMENTUM = 1e-5, 0.1
CONV_TOL = 2.0 ** -8
WGRAD_TOL = 1e-3
DOT_TOL = 1e-5


# ---------------------------------------------------------------------------------------------------------------------------
# fp64 per-layer references on NCHW tensors of logical pixels.  A conv layer is a valid conv over its padded input map.
def ref_pad(x, pad):
    return F.pad(x, (1, 1, 1, 1), mode="reflect") if pad else x


def ref_pad_adjoint(dp, pad):
    """Gradient w.r.t. the logical image of ref_pad: border rows / columns of dp add onto rows / columns 1 and H-2."""
    if not pad:
        return dp
    n, c, h, w = dp.shape
    x = torch.zeros((n, c, h - 2, w - 2), dtype=dp.dtype, device=dp.device, requires_grad=True)
    (g,) = torch.autograd.grad(F.pad(x, (1, 1, 1, 1), mode="reflect"), x, dp)
    return g


def ref_gate(act, slope):
    """LeakyReLU derivative from the sign of the stored activation (1 where there is no activation)."""
    if slope is None:
        return 1.0
    one = torch.ones((), dtype=torch.float64, device=act.device)
    return torch.where(act > 0, one, one * slope)


def ref_conv(p, w, b, slope, stride=1):
    y = F.conv2d(p, w, b, stride=stride)
    return y if slope is None else F.leaky_relu(y, slope)


def ref_conv_input_grad(g, w, in_shape, stride=1):
    return torch.nn.grad.conv2d_input(in_shape, w, g, stride=stride)


def ref_conv_weight_grad(p, g, w_shape, stride=1):
    """(dW, db) of the valid conv."""
    return torch.nn.grad.conv2d_weight(p, w_shape, g, stride=stride), g.sum(dim=(0, 2, 3))


def ref_bn_stats(x):
    """Batch mean and biased variance per channel."""
    return x.mean(dim=(0, 2, 3)), x.var(dim=(0, 2, 3), unbiased=False)


def ref_bn_train(x, gamma, beta):
    return F.batch_norm(x, None, None, gamma, beta, training=True, eps=EPS)


def ref_bn_backward(x, gamma, dy):
    """Autograd of the training-mode BatchNorm w.r.t. (x, gamma, beta)."""
    xr = x.detach().requires_grad_(True)
    gm = gamma.detach().clone().requires_grad_(True)
    bt = torch.zeros_like(gm, requires_grad=True)
    return torch.autograd.grad(ref_bn_train(xr, gm, bt), (xr, gm, bt), dy)


def ref_linear(x, w, b):
    return x @ w.t() + b


def ref_linear_backward(x, w, gy):
    """(dx, dW, db) of y = x W^T + b."""
    return gy @ w, gy.t() @ x, gy.sum(dim=0)


def _layers(d):
    from climsr_b200.models.discriminator import Discriminator
    return Discriminator._layers(d)


def ref_discriminator_forward(d, x, w_of=lambda m: m.weight.detach().double()):
    """The discriminator's forward chained from the per-layer references (BatchNorm in training mode)."""
    stages, conv4, conv5, lin0, lin1 = _layers(d)
    b_of = lambda m: m.bias.detach().double()                                 # noqa: E731
    acts, h = [], x
    for conv_a, bn, conv_b in stages:
        pa = ref_pad(h, 1)
        sa = ref_conv(pa, w_of(conv_a), b_of(conv_a), SLOPE)
        pb = ref_pad(ref_bn_train(sa, bn.weight.detach().double(), bn.bias.detach().double()), 1)
        sb = ref_conv(pb, w_of(conv_b), b_of(conv_b), SLOPE, stride=2)
        acts.append({"pa": pa, "sa": sa, "pb": pb, "sb": sb})
        h = sb
    s4 = ref_conv(h, w_of(conv4), b_of(conv4), SLOPE_TAIL)
    s5 = ref_conv(s4, w_of(conv5), b_of(conv5), None)
    feats = s5.reshape(s5.shape[0], -1)
    y1 = ref_linear(feats, lin0.weight.detach().double(), lin0.bias.detach().double())
    y2 = ref_linear(y1, lin1.weight.detach().double(), lin1.bias.detach().double())
    return {"stages": acts, "p4": h, "s4": s4, "s5": s5, "feats": feats, "y1": y1, "out": y2}


def ref_discriminator_backward(d, a, gy, w_of=lambda m: m.weight.detach().double()):
    """Input and parameter gradients chained from the per-layer references; {module: (dW, db)} and dx."""
    stages, conv4, conv5, lin0, lin1 = _layers(d)
    grads = {}
    dy1, dw, db = ref_linear_backward(a["y1"], lin1.weight.detach().double(), gy)
    grads[lin1] = (dw, db)
    dfeat, dw, db = ref_linear_backward(a["feats"], lin0.weight.detach().double(), dy1)
    grads[lin0] = (dw, db)
    g5 = dfeat.view(a["s5"].shape)
    grads[conv5] = ref_conv_weight_grad(a["s4"], g5, conv5.weight.shape)
    g4 = ref_conv_input_grad(g5, w_of(conv5), a["s4"].shape) * ref_gate(a["s4"], SLOPE_TAIL)
    grads[conv4] = ref_conv_weight_grad(a["p4"], g4, conv4.weight.shape)
    dp, pad_next = ref_conv_input_grad(g4, w_of(conv4), a["p4"].shape), 0
    for (conv_a, bn, conv_b), st in zip(reversed(stages), reversed(a["stages"])):
        gb = ref_pad_adjoint(dp, pad_next) * ref_gate(st["sb"], SLOPE)
        grads[conv_b] = ref_conv_weight_grad(st["pb"], gb, conv_b.weight.shape, stride=2)
        dpb = ref_conv_input_grad(gb, w_of(conv_b), st["pb"].shape, stride=2)
        dx_bn, dgamma, dbeta = ref_bn_backward(st["sa"], bn.weight.detach().double(), ref_pad_adjoint(dpb, 1))
        grads[bn] = (dgamma, dbeta)
        ga = dx_bn * ref_gate(st["sa"], SLOPE)
        grads[conv_a] = ref_conv_weight_grad(st["pa"], ga, conv_a.weight.shape)
        dp, pad_next = ref_conv_input_grad(ga, w_of(conv_a), st["pa"].shape), 1
    return ref_pad_adjoint(dp, 1), grads


# ---------------------------------------------------------------------------------------------------------------------------
# S-layout buffers and comparisons
def _view(t):
    from climsr_b200._lib import View
    return View(*t)


def _sl(v, n):
    return slice(v[3], v[3] + v[4] * n, v[4])


def _s_buffer(logical, v, fill=float("nan")):
    """(n, hs, ws, c) bf16 CUDA buffer holding `logical` (n, c, hl, wl) at its logical pixels and `fill` elsewhere."""
    hs, ws, c, off, step, hl, wl = v
    buf = torch.full((logical.shape[0], hs, ws, c), fill, dtype=torch.bfloat16, device="cuda")
    buf[:, _sl(v, hl), _sl(v, wl), :] = logical.permute(0, 2, 3, 1).to(device="cuda", dtype=torch.bfloat16)
    return buf


def _logical(buf, v):
    """(n, c, hl, wl) float64 of the logical pixels of an S-layout buffer."""
    return buf[:, _sl(v, v[5]), _sl(v, v[6]), :].permute(0, 3, 1, 2).double()


def _nchw(buf):
    return buf.permute(0, 3, 1, 2).double()


def _assert_zero_off_logical(buf, v, what):
    """Every pixel that is not logical holds +0 (bit pattern 0)."""
    mask = torch.ones((v[0], v[1]), dtype=torch.bool, device=buf.device)
    mask[_sl(v, v[5]), _sl(v, v[6])] = False
    bits = buf.view(torch.int16)[:, mask]
    assert bool((bits == 0).all()), f"{what}: non-logical pixels are not +0"


def _ulps(got, ref):
    """max |got - bf16(ref)| in units of the bf16 spacing at bf16(ref); NaN in `got` fails any bound."""
    rb = ref.to(torch.bfloat16).double()
    _, e = torch.frexp(rb)
    ulp = torch.where(rb == 0, torch.full_like(rb, 2.0 ** -133), torch.ldexp(torch.ones_like(rb), e - 8))
    return float(((got.double() - rb).abs() / ulp).max())


def _conv_err(got, ref):
    """Error of a conv-like output in units of its bound 2^-8 * max(1, max|ref|) (<= 1 passes)."""
    return float((got - ref).abs().max()) / (CONV_TOL * max(1.0, float(ref.abs().max())))


def _rel_l2(got, ref):
    return float((got - ref).norm() / ref.norm())


def _call(name, *args):
    from climsr_b200._lib import check, current_stream_ptr, lib
    check(getattr(lib, name)(*args, current_stream_ptr()), name)


def _bn_input(n, c, hl, wl, g):
    """Logical BatchNorm input, bf16-representable: channel c has mean 0, 10 or 100 times its standard deviation."""
    ratio = torch.tensor([0.0, 10.0, 100.0]).repeat(c)[:c].view(1, c, 1, 1)
    sigma = (torch.rand((1, c, 1, 1), generator=g) * 1.5 + 0.5)
    return (sigma * (ratio + torch.randn((n, c, hl, wl), generator=g))).to(torch.bfloat16).double()


def _signed_uniform(shape, g, lo=0.5, hi=1.5):
    mag = torch.rand(shape, generator=g) * (hi - lo) + lo
    return torch.where(torch.rand(shape, generator=g) < 0.5, -mag, mag)


# (n, view = (hs, ws, c, off, step, hl, wl), pad) of the glue kernels: the module's own views at batch 16, then the edges
GLUE_CASES = [
    (16, (128, 128, 64, 0, 1, 128, 128), 1),    # the input image (channel 0 of 64) -> stage 1 conv_a
    (16, (130, 130, 64, 1, 1, 128, 128), 1),    # stage 1 conv_a output -> BatchNorm -> conv_b
    (16, (130, 130, 64, 1, 2, 64, 64), 1),      # stage 1 stride-2 output -> stage 2
    (16, (66, 66, 128, 1, 1, 64, 64), 1),       # stage 2
    (16, (34, 34, 256, 1, 1, 32, 32), 1),       # stage 3
    (16, (18, 18, 512, 1, 1, 16, 16), 1),       # stage 4
    (16, (18, 18, 512, 1, 2, 8, 8), 0),         # stage 4 stride-2 output -> conv4 (valid)
    (16, (8, 8, 512, 1, 1, 6, 6), 0),           # conv4 -> conv5 (valid)
    (1, (4, 4, 8, 1, 1, 2, 2), 1),              # Hl = Wl = 2: both reflections land on every pixel; n = 1
    (3, (7, 7, 24, 1, 2, 3, 3), 1),             # Hl = Wl = 3: rows 1 and Hl-2 coincide; C = 24; stride 2
    (2, (6, 5, 8, 1, 1, 3, 2), 1),              # Hl != Wl
    (1, (11, 11, 512, 2, 2, 4, 4), 1),          # offset 2
]

# (n, view) of BatchNorm: the module's four at batch 16, then a stride-2 view and small / odd channel counts
BN_CASES = [
    (16, (130, 130, 64, 1, 1, 128, 128)),
    (16, (66, 66, 128, 1, 1, 64, 64)),
    (16, (34, 34, 256, 1, 1, 32, 32)),
    (16, (18, 18, 512, 1, 1, 16, 16)),
    (16, (130, 130, 64, 1, 2, 64, 64)),
    (1, (4, 4, 8, 1, 1, 2, 2)),
    (3, (7, 7, 24, 1, 2, 3, 3)),                # 24 channels: a 255-thread block
    (2, (10, 10, 512, 1, 1, 8, 8)),
]

# the ten convs: (name, padded input map, cin, cout, channels of the input buffer, LeakyReLU slope (0 = none))
LAYERS = [
    ("stage1.conv_a", 130, 1, 64, 64, SLOPE),
    ("stage1.conv_b", 130, 64, 64, 64, SLOPE),
    ("stage2.conv_a", 66, 64, 128, 64, SLOPE),
    ("stage2.conv_b", 66, 128, 128, 128, SLOPE),
    ("stage3.conv_a", 34, 128, 256, 128, SLOPE),
    ("stage3.conv_b", 34, 256, 256, 256, SLOPE),
    ("stage4.conv_a", 18, 256, 512, 256, SLOPE),
    ("stage4.conv_b", 18, 512, 512, 512, SLOPE),
    ("conv4", 8, 512, 512, 512, SLOPE_TAIL),
    ("conv5", 6, 512, 512, 512, 0.0),
]


def _ids(cases):
    return ["n%d-%s-p%d" % (c[0], "x".join(map(str, c[1])), c[2]) if len(c) > 2 else "n%d-%s" % (c[0], "x".join(map(str, c[1])))
            for c in cases]


# ---------------------------------------------------------------------------------------------------------------------------
# 1. glue kernels one at a time
@pytest.mark.gpu
@pytest.mark.parametrize("affine", [False, True], ids=["copy", "affine"])
@pytest.mark.parametrize("n,v,pad", GLUE_CASES, ids=_ids(GLUE_CASES))
def test_gather_matches_reflection_pad(n, v, pad, affine):
    hs, ws, c, off, step, hl, wl = v
    g = torch.Generator().manual_seed(hs * 7 + c + pad)
    x = torch.randn((n, c, hl, wl), generator=g).to(torch.bfloat16)
    src = _s_buffer(x, v)
    dst = torch.full((n, hl + 2 * pad, wl + 2 * pad, c), float("nan"), dtype=torch.bfloat16, device="cuda")
    scale = shift = None
    if affine:
        scale = torch.randn(c, generator=g).cuda()
        shift = (torch.randn(c, generator=g) * 3).cuda()
    _call("csr_disc_gather", src.data_ptr(), C.byref(_view(v)), n, dst.data_ptr(), pad,
          scale.data_ptr() if affine else None, shift.data_ptr() if affine else None)
    x64 = x.double().cuda()
    if affine:
        want = ref_pad(x64 * scale.double().view(1, c, 1, 1) + shift.double().view(1, c, 1, 1), pad)
        assert _ulps(_nchw(dst), want) <= 1.0
    else:
        assert torch.equal(_nchw(dst), ref_pad(x64, pad))


def _collect_case(n, v, pad, slope, seed):
    """Runs csr_disc_collect; returns (kernel output buffer, dP as float64 NCHW, act logical float64 or None)."""
    hs, ws, c, off, step, hl, wl = v
    g = torch.Generator().manual_seed(seed)
    dp = torch.randn((n, hl + 2 * pad, wl + 2 * pad, c), generator=g).to(torch.bfloat16).cuda()
    act = _s_buffer(torch.randn((n, c, hl, wl), generator=g), v) if slope is not None else None
    out = torch.full((n, hs, ws, c), float("nan"), dtype=torch.bfloat16, device="cuda")
    _call("csr_disc_collect", dp.data_ptr(), C.byref(_view(v)), n, pad, act.data_ptr() if act is not None else None,
          slope if slope is not None else 1.0, out.data_ptr())
    return out, _nchw(dp), (_logical(act, v) if act is not None else None)


@pytest.mark.gpu
@pytest.mark.parametrize("slope", [SLOPE, SLOPE_TAIL, None], ids=["slope0.01", "slope0.2", "noact"])
@pytest.mark.parametrize("n,v,pad", GLUE_CASES, ids=_ids(GLUE_CASES))
def test_collect_matches_reflection_pad_adjoint(n, v, pad, slope):
    out, dp, act = _collect_case(n, v, pad, slope, seed=v[0] + v[2] + pad)
    gate = ref_gate(act, slope)
    want = ref_pad_adjoint(dp, pad) * gate
    assert _ulps(_logical(out, v), want) <= 1.0
    _assert_zero_off_logical(out, v, "csr_disc_collect")
    if pad:
        # the bound sees the border terms: a reference without them (interior of dP only) is far outside it
        assert _ulps(_logical(out, v), dp[:, :, 1:-1, 1:-1] * gate) > 8.0


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["train", "train_no_running", "eval"])
@pytest.mark.parametrize("n,v", BN_CASES, ids=_ids(BN_CASES))
def test_bn_forward_statistics(n, v, mode):
    from climsr_b200._lib import lib
    hs, ws, c, off, step, hl, wl = v
    g = torch.Generator().manual_seed(c + hl + n)
    x = _bn_input(n, c, hl, wl, g)
    src = _s_buffer(x, v)
    gamma = _signed_uniform(c, g).cuda()
    beta = torch.randn(c, generator=g).cuda()
    rm0 = (torch.randn(c, generator=g) * 5).cuda()
    rv0 = (torch.rand(c, generator=g) * 2 + 0.5).cuda()
    rm, rv = rm0.clone(), rv0.clone()
    scale, shift, mean, invstd = (torch.full((c,), float("nan"), device="cuda") for _ in range(4))
    nbytes = lib.csr_disc_bn_scratch_bytes(c)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    running = mode != "train_no_running"
    _call("csr_disc_bn_forward", src.data_ptr(), C.byref(_view(v)), n, gamma.data_ptr(), beta.data_ptr(), EPS, MOMENTUM,
          rm.data_ptr() if running else None, rv.data_ptr() if running else None, 0 if mode == "eval" else 1, scale.data_ptr(),
          shift.data_ptr(), mean.data_ptr(), invstd.data_ptr(), scratch.data_ptr(), nbytes)
    g64, b64 = gamma.double(), beta.double()
    if mode == "eval":
        sc = g64 / torch.sqrt(rv0.double() + EPS)
        assert float(((scale.double() - sc).abs() / sc.abs()).max()) <= 1e-6                       # rsqrtf
        assert float(((shift.double() - (b64 - rm0.double() * sc)).abs() / (b64.abs() + (rm0.double() * sc).abs())).max()) <= 1e-6
        assert torch.equal(rm, rm0) and torch.equal(rv, rv0)
        return
    x64 = x.cuda()
    m_ref, var_ref = ref_bn_stats(x64)
    std_ref = var_ref.sqrt()
    inv_ref = 1.0 / torch.sqrt(var_ref + EPS)
    # the mean of a zero-mean channel is itself rounding noise: its error is measured against |mean| + std
    assert float(((mean.double() - m_ref).abs() / (m_ref.abs() + std_ref)).max()) <= 1e-4
    assert float(((invstd.double() - inv_ref).abs() / inv_ref).max()) <= 1e-4
    # what the finalisation computes from those statistics
    mk, ik = mean.double(), invstd.double()
    sc = g64 * ik
    assert float(((scale.double() - sc).abs() / sc.abs()).max()) <= 1e-5
    assert float(((shift.double() - (b64 - mk * sc)).abs() / (b64.abs() + (mk * sc).abs())).max()) <= 1e-5
    if running:
        m_cnt = n * hl * wl
        var_k = 1.0 / (ik * ik) - EPS                                                            # the variance behind invstd
        want_m = (1 - MOMENTUM) * rm0.double() + MOMENTUM * mk
        want_v = (1 - MOMENTUM) * rv0.double() + MOMENTUM * var_k * m_cnt / max(m_cnt - 1, 1)
        assert float(((rm.double() - want_m).abs() / ((1 - MOMENTUM) * rm0.double().abs() + MOMENTUM * mk.abs())).max()) <= 1e-5
        assert float(((rv.double() - want_v).abs() / want_v.abs()).max()) <= 1e-5
    else:
        assert torch.equal(rm, rm0) and torch.equal(rv, rv0)


BN_BWD_CASES = [(n, v, 1) for n, v in BN_CASES] + [(2, (8, 8, 24, 1, 1, 6, 6), 0)]


def bn_backward_case(n, v, pad, seed=0):
    """Runs csr_disc_bn_backward on an upstream gradient dP = a_c + b_c * reflect_pad(xhat) + noise (a_c, b_c of the noise's
    order, so both correction terms of the backward carry most of the answer).  Returns the errors of the kernel against the
    fp64 reference and against references that drop either correction term."""
    from climsr_b200._lib import lib
    hs, ws, c, off, step, hl, wl = v
    g = torch.Generator().manual_seed(seed + c + hl)
    x = _bn_input(n, c, hl, wl, g).cuda()
    m64, var64 = ref_bn_stats(x)
    mean_k, invstd_k = m64.float(), (1.0 / torch.sqrt(var64 + EPS)).float()          # what the forward hands the backward
    xhat_p = ref_pad((x - m64.view(1, c, 1, 1)) / torch.sqrt(var64 + EPS).view(1, c, 1, 1), pad)
    a = _signed_uniform((1, c, 1, 1), g).double().cuda()
    b = _signed_uniform((1, c, 1, 1), g).double().cuda()
    dp = (a + b * xhat_p + torch.randn(xhat_p.shape, generator=g, dtype=torch.float64).cuda()).to(torch.bfloat16)
    dp_buf = dp.permute(0, 2, 3, 1).contiguous()
    gamma = _signed_uniform(c, g).cuda()
    act = _s_buffer(x, v)
    dy_scratch = torch.full((n * hl * wl * c,), float("nan"), device="cuda")
    nbytes = lib.csr_disc_bn_scratch_bytes(c)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    out = torch.full((n, hs, ws, c), float("nan"), dtype=torch.bfloat16, device="cuda")
    dgamma = torch.ones(c, device="cuda")
    dbeta = torch.ones(c, device="cuda")
    _call("csr_disc_bn_backward", dp_buf.data_ptr(), C.byref(_view(v)), n, pad, act.data_ptr(), SLOPE, gamma.data_ptr(),
          mean_k.data_ptr(), invstd_k.data_ptr(), dy_scratch.data_ptr(), scratch.data_ptr(), nbytes, out.data_ptr(), dgamma.data_ptr(),
          dbeta.data_ptr())
    dy = ref_pad_adjoint(dp.double(), pad)
    dx, _, _ = ref_bn_backward(x, gamma.double(), dy)
    gate = ref_gate(x, SLOPE)
    want = dx * gate
    got = _logical(out, v)
    # dgamma / dbeta from the statistics the kernel was given (fp32 mean / invstd)
    xhat_k = (x - mean_k.double().view(1, c, 1, 1)) * invstd_k.double().view(1, c, 1, 1)
    dgamma_ref, dbeta_ref = (dy * xhat_k).sum(dim=(0, 2, 3)), dy.sum(dim=(0, 2, 3))
    # the two correction terms, each dropped in turn from the analytic form gamma * invstd * (dy - mean(dy) - xhat * mean(dy xhat))
    k = gamma.double().view(1, c, 1, 1) * invstd_k.double().view(1, c, 1, 1)
    mean_dy = dy.mean(dim=(0, 2, 3), keepdim=True)
    mean_dyx = (dy * xhat_k).mean(dim=(0, 2, 3), keepdim=True)
    no_mean_term = k * (dy - xhat_k * mean_dyx) * gate
    no_xhat_term = k * (dy - mean_dy) * gate
    return {
        "out": out, "v": v,
        "rel_l2": _rel_l2(got, want), "max": float((got - want).abs().max()) / float(want.abs().max()),
        "dgamma": float((((dgamma.double() - 1) - dgamma_ref).abs() / dgamma_ref.abs()).max()),
        "dbeta": float((((dbeta.double() - 1) - dbeta_ref).abs() / dbeta_ref.abs()).max()),
        "rel_l2_without_mean_term": _rel_l2(got, no_mean_term), "rel_l2_without_xhat_term": _rel_l2(got, no_xhat_term),
    }


@pytest.mark.gpu
@pytest.mark.parametrize("n,v,pad", BN_BWD_CASES, ids=_ids(BN_BWD_CASES))
def test_bn_backward_matches_autograd(n, v, pad):
    r = bn_backward_case(n, v, pad)
    assert r["rel_l2"] <= 3e-3 and r["max"] <= 2.0 ** -7, r
    assert r["dgamma"] <= 1e-5 and r["dbeta"] <= 1e-5, r
    _assert_zero_off_logical(r["out"], v, "csr_disc_bn_backward")
    # the bound sees both correction terms: references without either are far outside it
    assert r["rel_l2_without_mean_term"] > 0.1 and r["rel_l2_without_xhat_term"] > 0.1, r


FLAT_CASES = [(16, (6, 6, 512, 1, 1, 4, 4)), (1, (6, 6, 512, 1, 1, 4, 4)), (3, (7, 7, 24, 1, 2, 3, 3)), (2, (5, 4, 8, 0, 1, 5, 4))]


@pytest.mark.gpu
@pytest.mark.parametrize("n,v", FLAT_CASES, ids=_ids(FLAT_CASES))
def test_flatten_and_unflatten(n, v):
    hs, ws, c, off, step, hl, wl = v
    g = torch.Generator().manual_seed(n + c)
    x = torch.randn((n, c, hl, wl), generator=g).to(torch.bfloat16)
    feats = torch.full((n, c * hl * wl), float("nan"), device="cuda")
    _call("csr_disc_flatten", _s_buffer(x, v).data_ptr(), C.byref(_view(v)), n, feats.data_ptr())
    assert torch.equal(feats.cpu(), x.float().view(n, -1))                  # x.view(N, -1) of the NCHW logical tensor
    gfeat = torch.randn((n, c * hl * wl), generator=g).cuda()
    out = torch.full((n, hs, ws, c), float("nan"), dtype=torch.bfloat16, device="cuda")
    _call("csr_disc_unflatten", gfeat.data_ptr(), C.byref(_view(v)), n, out.data_ptr())
    want = _s_buffer(gfeat.view(n, c, hl, wl), v, fill=0.0)
    assert torch.equal(out.view(torch.int16), want.view(torch.int16))
    _assert_zero_off_logical(out, v, "csr_disc_unflatten")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 16, 65])
@pytest.mark.parametrize("k,j", [(8192, 100), (100, 1)])
def test_linear_forward_and_backward(n, k, j):
    g = torch.Generator().manual_seed(n + k)
    x = torch.randn((n, k), generator=g).cuda()
    w = (torch.randn((j, k), generator=g) / k ** 0.5).cuda()
    b = torch.randn(j, generator=g).cuda()
    gy = torch.randn((n, j), generator=g).cuda()
    x64, w64, b64, gy64 = x.double(), w.double(), b.double(), gy.double()
    y = torch.full((n, j), float("nan"), device="cuda")
    _call("csr_linear_forward", x.data_ptr(), w.data_ptr(), b.data_ptr(), y.data_ptr(), n, k, j)
    assert bool(((y.double() - ref_linear(x64, w64, b64)).abs() <= DOT_TOL * (x64.abs() @ w64.abs().t() + b64.abs())).all())
    dx_ref, dw_ref, db_ref = ref_linear_backward(x64, w64, gy64)
    dx_tol = DOT_TOL * (gy64.abs() @ w64.abs())
    # accumulating outputs start at 1: the fp32 rounding of 1 + sum adds half an ulp of the result
    dw_tol = DOT_TOL * (gy64.abs().t() @ x64.abs()) + 2.0 ** -24 * (1 + dw_ref).abs()
    db_tol = DOT_TOL * gy64.abs().sum(dim=0) + 2.0 ** -24 * (1 + db_ref).abs()
    for want_dx, want_dw, want_db in ((1, 1, 1), (0, 1, 1), (1, 0, 1), (1, 1, 0), (0, 0, 1)):
        dx = torch.full((n, k), float("nan"), device="cuda") if want_dx else None
        dw = torch.ones((j, k), device="cuda") if want_dw else None
        db = torch.ones(j, device="cuda") if want_db else None
        _call("csr_linear_backward", x.data_ptr(), w.data_ptr(), gy.data_ptr(), dx.data_ptr() if want_dx else None,
              dw.data_ptr() if want_dw else None, db.data_ptr() if want_db else None, n, k, j)
        what = (want_dx, want_dw, want_db)
        if want_dx:
            assert bool(((dx.double() - dx_ref).abs() <= dx_tol).all()), what
        if want_dw:
            assert bool(((dw.double() - 1 - dw_ref).abs() <= dw_tol).all()), what
        if want_db:
            assert bool(((db.double() - 1 - db_ref).abs() <= db_tol).all()), what


# ---------------------------------------------------------------------------------------------------------------------------
# 2. the ten convs: prepacked weights, transposed (input-gradient) convs
@pytest.mark.gpu
@pytest.mark.parametrize("name,hp,cin,cout,in_c,slope", LAYERS, ids=[l[0] for l in LAYERS])
def test_layer_prepacked_and_transposed(name, hp, cin, cout, in_c, slope):
    from climsr_b200 import ops
    n = 16
    g = torch.Generator().manual_seed(hp + cin + cout)
    wt = ((torch.rand((cout, cin, 3, 3), generator=g) * 2 - 1) / (cin * 9) ** 0.5).cuda()
    b = (torch.rand((cout,), generator=g) - 0.5).cuda()
    x = torch.zeros((n, hp, hp, in_c), dtype=torch.bfloat16, device="cuda")
    x[..., :cin] = (torch.rand((n, hp, hp, cin), generator=g) * 2 - 1).to(torch.bfloat16).cuda()
    act = dict(act="lrelu_slope", act_slope=slope) if slope else dict(act="none")
    # the module packs each layer once (csr_conv2d_pack) and runs it prepacked: the same bits as packing inside the call
    fwd = ops.conv2d_nhwc(x, wt, b, out=torch.full((n, hp, hp, cout), float("nan"), dtype=torch.bfloat16, device="cuda"), **act)
    scratch = torch.empty(max(ops.conv2d_scratch_bytes(cout, cin, 3, 3, False), 16), dtype=torch.uint8, device="cuda")
    ops.conv2d_pack(wt, b, scratch, False)
    pre = ops.conv2d_nhwc(x, wt, b, out=torch.full((n, hp, hp, cout), float("nan"), dtype=torch.bfloat16, device="cuda"),
                          scratch=scratch, prepacked=True, **act)
    assert torch.equal(fwd, pre), name
    # input gradient: the transposed conv over a gradient map defined at every pixel, against the fp64 adjoint
    gy = (torch.rand((n, hp, hp, cout), generator=g) * 2 - 1).to(torch.bfloat16).cuda()
    oc = (cin + 63) // 64 * 64
    dx = ops.conv2d_nhwc(gy, wt, None, transposed=True, out=torch.full((n, hp, hp, oc), float("nan"), dtype=torch.bfloat16, device="cuda"))
    want = F.conv_transpose2d(_nchw(gy), wt.to(torch.bfloat16).double(), padding=1)
    assert _conv_err(_nchw(dx[..., :cin]), want) <= 1.0, name
    tscratch = torch.empty(max(ops.conv2d_scratch_bytes(cin, cout, 3, 3, True), 16), dtype=torch.uint8, device="cuda")
    ops.conv2d_pack(wt, None, tscratch, True)
    dx_pre = ops.conv2d_nhwc(gy, wt, None, transposed=True, scratch=tscratch, prepacked=True,
                             out=torch.full((n, hp, hp, oc), float("nan"), dtype=torch.bfloat16, device="cuda"))
    assert torch.equal(dx[..., :cin], dx_pre[..., :cin]), name


# ---------------------------------------------------------------------------------------------------------------------------
# 3. the module, layer by layer, at batch 16: every layer against the fp64 reference of its own stored inputs
def _make(seed):
    from climsr_b200.models.discriminator import Discriminator
    from oracle import synth
    d = Discriminator()
    d.load_state_dict(synth.make_discriminator_state_dict(seed=seed), strict=True)
    return d


class _Capture:
    """Records the arguments and results of the module-level layer helpers of climsr_b200.models.discriminator."""
    NAMES = ("_gather", "_conv", "_collect", "_conv_t", "_wgrad")

    def __init__(self):
        from climsr_b200.models import discriminator as D
        self.D, self.orig, self.rec = D, {k: getattr(D, k) for k in self.NAMES}, {k: [] for k in self.NAMES}

    def __enter__(self):
        for k in self.NAMES:
            setattr(self.D, k, self._wrap(k))
        return self.rec

    def _wrap(self, k):
        f = self.orig[k]

        def spy(*args):
            out = f(*args)
            self.rec[k].append((args, out))
            return out
        return spy

    def __exit__(self, *exc):
        for k, f in self.orig.items():
            setattr(self.D, k, f)


def _vt(view):
    return (view.hs, view.ws, view.c, view.off, view.step, view.hl, view.wl)


def _wbf(m):
    return m.weight.detach().to(torch.bfloat16).double()


def _check_forward(d, x, rec, training, rm0, rv0, saved=None):
    """Each forward layer against the fp64 reference of the operands the kernels stored."""
    stages, conv4, conv5, lin0, lin1 = _layers(d)
    gathers, convs = rec["_gather"], rec["_conv"]
    assert len(gathers) == 10 and len(convs) == 10
    n = x.shape[0]
    # the input image: channel 0 of a 64-channel bf16 buffer
    src0 = gathers[0][0][0]
    assert torch.equal(_nchw(src0)[:, :1], x.to(torch.bfloat16).double()) and not bool(src0[..., 1:].any())
    for i, ((conv_a, bn, conv_b), gi) in enumerate(zip(stages, range(0, 8, 2))):
        (src, view, _, pad), pa = gathers[gi][0][:4], gathers[gi][1]
        assert torch.equal(_nchw(pa), ref_pad(_logical(src, _vt(view)), pad)), i
        (p, _, _, slope, _), sa = convs[gi]
        assert p is pa and slope == SLOPE
        cin = conv_a.in_channels
        want = ref_conv(_nchw(pa)[:, :cin], _wbf(conv_a), conv_a.bias.detach().double(), SLOPE)
        va = (view.hl + 2, view.wl + 2, conv_a.out_channels, 1, 1, view.hl, view.wl)
        assert _conv_err(_logical(sa, va), want) <= 1.0, (i, "conv_a")
        (src_b, view_b, _, _, scale, shift), pb = gathers[gi + 1]
        assert src_b is sa and _vt(view_b) == va
        g64, b64 = bn.weight.detach().double(), bn.bias.detach().double()
        xs = _logical(sa, va)
        if training:
            m_ref, var_ref = ref_bn_stats(xs)
            mean, invstd = saved["stages"][i]["mean"], saved["stages"][i]["invstd"]
            assert float(((mean.double() - m_ref).abs() / (m_ref.abs() + var_ref.sqrt())).max()) <= 1e-4, i
            inv_ref = 1.0 / torch.sqrt(var_ref + EPS)
            assert float(((invstd.double() - inv_ref).abs() / inv_ref).max()) <= 1e-4, i
            mk, ik = mean.double(), invstd.double()
            sc = g64 * ik
            assert float(((scale.double() - sc).abs() / sc.abs()).max()) <= 1e-5, i
            assert float(((shift.double() - (b64 - mk * sc)).abs() / (b64.abs() + (mk * sc).abs())).max()) <= 1e-5, i
            m_cnt = n * va[5] * va[6]
            want_m = (1 - MOMENTUM) * rm0[i] + MOMENTUM * mk
            want_v = (1 - MOMENTUM) * rv0[i] + MOMENTUM * (1.0 / (ik * ik) - EPS) * m_cnt / (m_cnt - 1)
            assert float(((bn.running_mean.double() - want_m).abs() / ((1 - MOMENTUM) * rm0[i].abs() + MOMENTUM * mk.abs())).max()) <= 1e-5, i
            assert float(((bn.running_var.double() - want_v).abs() / want_v).max()) <= 1e-5, i
        else:
            sc = g64 / torch.sqrt(bn.running_var.double() + EPS)
            assert float(((scale.double() - sc).abs() / sc.abs()).max()) <= 1e-6, i
            rms = bn.running_mean.double() * sc
            assert float(((shift.double() - (b64 - rms)).abs() / (b64.abs() + rms.abs())).max()) <= 1e-6, i
            assert torch.equal(bn.running_mean.double(), rm0[i]) and torch.equal(bn.running_var.double(), rv0[i]), i
        c = bn.num_features
        affine = xs * scale.double().view(1, c, 1, 1) + shift.double().view(1, c, 1, 1)
        assert _ulps(_nchw(pb), ref_pad(affine, 1)) <= 1.0, (i, "BatchNorm gather")
        (p, _, _, slope, _), sb = convs[gi + 1]
        assert p is pb and slope == SLOPE
        want = ref_conv(_nchw(pb), _wbf(conv_b), conv_b.bias.detach().double(), SLOPE, stride=2)
        vb = (va[0], va[1], c, 1, 2, va[5] // 2, va[6] // 2)
        assert _conv_err(_logical(sb, vb), want) <= 1.0, (i, "conv_b")
    (src4, view4, _, pad4), p4 = gathers[8][0][:4], gathers[8][1]
    assert pad4 == 0 and torch.equal(_nchw(p4), _logical(src4, _vt(view4)))
    (_, _, _, slope4, _), s4 = convs[8]
    assert slope4 == SLOPE_TAIL
    v4 = (8, 8, 512, 1, 1, 6, 6)
    assert _conv_err(_logical(s4, v4), ref_conv(_nchw(p4), _wbf(conv4), conv4.bias.detach().double(), SLOPE_TAIL)) <= 1.0, "conv4"
    (src5, view5, _, pad5), p5 = gathers[9][0][:4], gathers[9][1]
    assert src5 is s4 and _vt(view5) == v4 and pad5 == 0 and torch.equal(_nchw(p5), _logical(s4, v4))
    (_, _, _, slope5, _), s5 = convs[9]
    assert slope5 == 0.0
    v5 = (6, 6, 512, 1, 1, 4, 4)
    assert _conv_err(_logical(s5, v5), ref_conv(_nchw(p5), _wbf(conv5), conv5.bias.detach().double(), None)) <= 1.0, "conv5"
    return s5, v5


def _check_head(d, s5, v5, saved, out):
    """flatten + the two Linear layers."""
    _, _, _, lin0, lin1 = _layers(d)
    n = s5.shape[0]
    feats = _logical(s5, v5).reshape(n, -1)
    w0, b0, w1, b1 = (t.detach().double() for t in (lin0.weight, lin0.bias, lin1.weight, lin1.bias))
    if saved is not None:
        assert torch.equal(saved["feats"].double(), feats)
        y1 = saved["y1"].double()
        assert bool(((y1 - ref_linear(feats, w0, b0)).abs() <= DOT_TOL * (feats.abs() @ w0.abs().t() + b0.abs())).all())
        assert bool(((out.double() - ref_linear(y1, w1, b1)).abs() <= DOT_TOL * (y1.abs() @ w1.abs().t() + b1.abs())).all())
    else:                                                           # y1 not kept: its bound carried through the second layer
        y1 = ref_linear(feats, w0, b0)
        e1 = DOT_TOL * (feats.abs() @ w0.abs().t() + b0.abs())
        tol = DOT_TOL * ((y1.abs() + e1) @ w1.abs().t() + b1.abs()) + e1 @ w1.abs().t()
        assert bool(((out.double() - ref_linear(y1, w1, b1)).abs() <= tol).all())


def _check_backward(d, saved, gy, dx, grads, rec, need_params):
    """Each backward layer against the fp64 reference of the operands the kernels stored."""
    stages, conv4, conv5, lin0, lin1 = _layers(d)
    n = saved["n"]
    convt, coll, wg = rec["_conv_t"], rec["_collect"], rec["_wgrad"]
    assert len(convt) == 10 and len(coll) == 6 and len(wg) == (10 if need_params else 0)
    by_mod = dict(zip(d._module_order(), zip(grads[0::2], grads[1::2])))
    gy64 = gy.double()
    w0, w1 = lin0.weight.detach().double(), lin1.weight.detach().double()
    y1, feats = saved["y1"].double(), saved["feats"].double()
    # linear backward, unflatten
    dy1_ref, dw1_ref, db1_ref = ref_linear_backward(y1, w1, gy64)
    e_dy1 = DOT_TOL * (gy64.abs() @ w1.abs())
    dfeat_ref, dw0_ref, db0_ref = ref_linear_backward(feats, w0, dy1_ref)
    e_dfeat = DOT_TOL * ((dy1_ref.abs() + e_dy1) @ w0.abs()) + e_dy1 @ w0.abs()
    (g5, _, _), dp5 = convt[0]
    v5 = _vt(saved["v5"])
    got5 = _logical(g5, v5).reshape(n, -1)
    rb = dfeat_ref.to(torch.bfloat16).double()
    _, e = torch.frexp(rb)
    assert bool(((got5 - dfeat_ref).abs() <= torch.ldexp(torch.ones_like(rb), e - 8) + e_dfeat).all()), "unflatten(linear backward)"
    _assert_zero_off_logical(g5, v5, "unflatten")
    if need_params:
        dw1, db1 = by_mod[lin1]
        assert bool(((dw1.double() - dw1_ref).abs() <= DOT_TOL * (gy64.abs().t() @ y1.abs())).all())
        assert bool(((db1.double() - db1_ref).abs() <= DOT_TOL * gy64.abs().sum(dim=0)).all())
        dw0, db0 = by_mod[lin0]
        e_w0 = DOT_TOL * ((dy1_ref.abs() + e_dy1).t() @ feats.abs()) + e_dy1.t() @ feats.abs()
        assert bool(((dw0.double() - dw0_ref).abs() <= e_w0).all())
        assert bool(((db0.double() - db0_ref).abs() <= DOT_TOL * (dy1_ref.abs() + e_dy1).sum(dim=0) + e_dy1.sum(dim=0)).all())
    else:
        assert all(by_mod[m] == (None, None) for m in (lin0, lin1, conv4, conv5))

    def conv_layer(conv, p, g, view, stride, idx, what):
        """Input gradient (and weight gradient) of one conv from its stored input map p and its gradient g, logical at `view`
        (the S-layout gradient is zero elsewhere, so the kernels' same-convs over the padded map are the valid conv's adjoints)."""
        (gg, _, _), dp = convt[idx]
        assert gg is g, what
        cin = conv.in_channels
        p64, g64 = _nchw(p)[:, :cin], _logical(g, view)
        want = ref_conv_input_grad(g64, _wbf(conv), p64.shape, stride)
        assert _conv_err(_nchw(dp)[:, :cin], want) <= 1.0, (what, "input gradient")
        if need_params:
            (pp, gw, _, _), (dw, db) = wg[idx]
            assert pp is p and gw is g, what
            dw_ref, db_ref = ref_conv_weight_grad(p64, g64, conv.weight.shape, stride)
            assert by_mod[conv][0] is dw and by_mod[conv][1] is db, what
            ew = float((dw.double() - dw_ref).abs().max()) / float(dw_ref.abs().max())
            eb = float((db.double() - db_ref).abs().max()) / float(db_ref.abs().max())
            assert ew <= WGRAD_TOL and eb <= WGRAD_TOL, (what, ew, eb)
        return dp

    def collect(k, dp, view, pad, act, slope, what):
        (dpp, vw, _, pp, a, gate_neg), g = coll[k]
        assert dpp is dp and _vt(vw) == view and pp == pad and a is act, what
        assert gate_neg == (slope if slope is not None else 1.0), what
        want = ref_pad_adjoint(_nchw(dp), pad) * ref_gate(_logical(act, view) if act is not None else None, slope)
        assert _ulps(_logical(g, view), want) <= 1.0, what
        _assert_zero_off_logical(g, view, what)
        return g

    dp5 = conv_layer(conv5, saved["p5"], g5, v5, 1, 0, "conv5")
    v4 = _vt(saved["v4"])
    g4 = collect(0, dp5, v4, 0, saved["s4"], SLOPE_TAIL, "conv4 gate")
    dp = conv_layer(conv4, saved["p4"], g4, v4, 1, 1, "conv4")
    pad_next = 0
    for k, ((conv_a, bn, conv_b), st) in enumerate(zip(reversed(stages), reversed(saved["stages"]))):
        i = len(stages) - 1 - k
        gb = collect(1 + k, dp, _vt(st["vb"]), pad_next, st["sb"], SLOPE, f"stage {i + 1} conv_b gate")
        dpb = conv_layer(conv_b, st["pb"], gb, _vt(st["vb"]), 2, 2 + 2 * k, f"stage {i + 1} conv_b")
        # BatchNorm backward: its output is the gradient conv_a's input-gradient conv reads
        va = _vt(st["va"])
        ga = convt[3 + 2 * k][0][0]
        x = _logical(st["sa"], va)
        c = bn.num_features
        dy = ref_pad_adjoint(_nchw(dpb), 1)
        dxb, _, _ = ref_bn_backward(x, bn.weight.detach().double(), dy)
        want = dxb * ref_gate(x, SLOPE)
        got = _logical(ga, va)
        assert _rel_l2(got, want) <= 3e-3 and float((got - want).abs().max()) <= 2.0 ** -7 * float(want.abs().max()), (i, "BatchNorm backward")
        _assert_zero_off_logical(ga, va, f"stage {i + 1} BatchNorm backward")
        xhat_k = (x - st["mean"].double().view(1, c, 1, 1)) * st["invstd"].double().view(1, c, 1, 1)
        # dgamma / dbeta are sums over 262 144 ... 4 096 products that need not share a sign: measured against the sum of
        # their magnitudes, the fp32 summation bound
        dgamma, dbeta = by_mod[bn]
        prod = dy * xhat_k
        assert float(((dgamma.double() - prod.sum(dim=(0, 2, 3))).abs() / prod.abs().sum(dim=(0, 2, 3))).max()) <= 1e-5, i
        assert float(((dbeta.double() - dy.sum(dim=(0, 2, 3))).abs() / dy.abs().sum(dim=(0, 2, 3))).max()) <= 1e-5, i
        dp = conv_layer(conv_a, st["pa"], ga, va, 1, 3 + 2 * k, f"stage {i + 1} conv_a")
        pad_next = 1
    v0 = (128, 128, 64, 0, 1, 128, 128)
    gx = collect(5, dp, v0, 1, None, None, "input gradient")
    assert torch.equal(dx.double(), _nchw(gx)[:, :1])


def _module_case(seed, n):
    d = _make(seed).cuda().train()
    g = torch.Generator().manual_seed(seed + 100)
    x = (torch.rand((n, 1, 128, 128), generator=g) * 2 - 1).cuda()
    gy = torch.randn((n, 1), generator=g).cuda()
    bns = [st[1] for st in _layers(d)[0]]
    with torch.no_grad():                                    # non-trivial running statistics
        for bn in bns:
            bn.running_mean.copy_(torch.randn(bn.num_features, generator=g))
            bn.running_var.copy_(torch.rand(bn.num_features, generator=g) + 0.5)
    return d, x, gy, bns


@pytest.mark.gpu
def test_module_layer_by_layer_at_batch_16():
    """Training mode: the forward with every BatchNorm on batch statistics, then the backward with all gradients and the frozen
    backward (input gradient only, as the generator's adversarial loss runs it) on the same saved forward."""
    d, x, gy, bns = _module_case(seed=4, n=16)
    rm0 = [bn.running_mean.double().clone() for bn in bns]
    rv0 = [bn.running_var.double().clone() for bn in bns]
    with _Capture() as rec, torch.no_grad():
        out, saved = d._run_forward(x, save=True)
    s5, v5 = _check_forward(d, x, rec, True, rm0, rv0, saved)
    _check_head(d, s5, v5, saved, out)
    for need_params in (True, False):
        with _Capture() as rec, torch.no_grad():
            dx, grads = d._run_backward(saved, gy, True, need_params)
        _check_backward(d, saved, gy, dx, grads, rec, need_params)


@pytest.mark.gpu
def test_module_layer_by_layer_eval_forward():
    """Eval mode: BatchNorm from the running statistics, which the forward leaves untouched."""
    d, x, _, bns = _module_case(seed=6, n=16)
    d.eval()
    rm0 = [bn.running_mean.double().clone() for bn in bns]
    rv0 = [bn.running_var.double().clone() for bn in bns]
    with _Capture() as rec, torch.no_grad():
        out, saved = d._run_forward(x, save=False)
    assert saved is None
    s5, v5 = _check_forward(d, x, rec, False, rm0, rv0)
    _check_head(d, s5, v5, None, out)


# ---------------------------------------------------------------------------------------------------------------------------
# 4. BatchNorm momentum
@pytest.mark.gpu
def test_batchnorm_momentum_none_is_rejected_in_training():
    from climsr_b200._lib import CsrError
    d = _make(seed=0).cuda().train()
    x = (torch.rand((2, 1, 128, 128)) * 2 - 1).cuda()
    bn = _layers(d)[0][1][1]
    bn.momentum = None                                       # PyTorch: cumulative moving average
    with pytest.raises(CsrError, match="momentum=None"):
        d(x)
    with pytest.raises(CsrError, match="momentum=None"), torch.no_grad():
        d(x)
    assert int(bn.num_batches_tracked) == 0                  # rejected before anything ran
    d.eval()                                                 # eval mode reads the running statistics: momentum is unused
    with torch.no_grad():
        assert bool(torch.isfinite(d(x)).all())


@pytest.mark.gpu
def test_momentum_change_reaches_graph_replays():
    """Graph replays bake the momentum into the captured launches: a changed momentum must not replay a stale graph."""
    d = _make(seed=1).cuda().train()
    e = copy.deepcopy(d)
    e.use_cuda_graphs = False
    x = (torch.rand((2, 1, 128, 128)) * 2 - 1).cuda()
    with torch.no_grad():
        for _ in range(3):                                   # the third call replays a graph
            d(x), e(x)
        for m in (d, e):
            for st in _layers(m)[0]:
                st[1].momentum = 0.5
        for _ in range(3):
            d(x), e(x)
    for (name, a), (_, b) in zip(d.named_buffers(), e.named_buffers()):
        assert float((a.double() - b.double()).abs().max()) <= 1e-4 * max(1.0, float(b.double().abs().max())), name


# ---------------------------------------------------------------------------------------------------------------------------
# the references themselves (CPU)
def test_reference_chain_reproduces_stock_pytorch():
    """The fp64 per-layer references above, chained with no rounding, give stock PyTorch's forward and autograd gradients of
    the module's own containers (feature_extraction / classification) to 1e-10."""
    from oracle import synth
    from climsr_b200.models.discriminator import Discriminator
    d = Discriminator()
    d.load_state_dict(synth.make_discriminator_state_dict(seed=2), strict=True)
    d = d.double().train()
    g = torch.Generator().manual_seed(3)
    x = (torch.rand((2, 1, 128, 128), generator=g, dtype=torch.float64) * 2 - 1)
    gy = torch.randn((2, 1), generator=g, dtype=torch.float64)
    ref = copy.deepcopy(d)
    xr = x.clone().requires_grad_(True)
    f = ref.feature_extraction(xr)
    out = ref.classification(f.view(f.size(0), -1))
    out.backward(gy)
    w_of = lambda m: m.weight.detach()                                          # noqa: E731
    with torch.no_grad():
        a = ref_discriminator_forward(d, x, w_of)
    assert float((a["out"] - out.detach()).abs().max()) <= 1e-10 * float(out.detach().abs().max())
    dx, grads = ref_discriminator_backward(d, a, gy, w_of)
    assert float((dx - xr.grad).abs().max()) <= 1e-10 * float(xr.grad.abs().max())
    mods_ref = dict(zip(d._module_order(), ref._module_order()))
    assert len(grads) == len(mods_ref) == 16
    for m, (gw, gb) in grads.items():
        r = mods_ref[m]
        for got, want in ((gw, r.weight.grad), (gb, r.bias.grad)):
            assert float((got - want).abs().max()) <= 1e-10 * float(want.abs().max()), type(m).__name__
