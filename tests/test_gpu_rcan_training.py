"""GPU tests of RCAN training (SURVEY.md section 8f row 4): the channel-attention backward and PixelUnshuffle kernels, the conv
shapes only the RCAN backward uses, and the whole autograd path against the reference's golden gradients and the fp32 oracle.

Tolerances.  Single kernels are held to the rounding of their own operands: <= 1e-3 relative on exact operands, 2^-7 of the
largest reference value on bf16 outputs.  The whole backward stores every activation and gradient map in bf16, so it is held
to cosine and relative L2 bounds set at about twice the worst tensor measured on an NVIDIA B200 (the measured worsts are
next to the bounds).
"""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

GEN_TOL = 1e-2          # generator max-abs error in normalised units (the forward parity tolerance)


def _bf(t):
    return t.to(torch.bfloat16).float()


def _nhwc(x, c=64, fill=0.0):
    out = torch.full((x.shape[0], x.shape[2], x.shape[3], c), fill, dtype=torch.bfloat16)
    out[..., :x.shape[1]] = x.permute(0, 2, 3, 1).to(torch.bfloat16)
    return out.cuda()


def _nchw(t, c):
    return t[..., :c].float().cpu().permute(0, 3, 1, 2)


def _rcan(ng, nbk, seed):
    from climsr_b200.models.rcan import RCAN
    torch.manual_seed(seed)
    return RCAN(n_resgroups=ng, n_resblocks=nbk, n_feats=64, reduction=16, scaling_factor=4, in_channels=3, out_channels=1)


def _metrics(g, ref):
    g, ref = g.flatten().double(), ref.flatten().double()
    rel = float((g - ref).norm() / (ref.norm() + 1e-30))
    cos = float(F.cosine_similarity(g, ref, dim=0)) if float(ref.norm()) > 0 else 1.0
    return rel, cos


# ---------------------------------------------------------------------------------------------------- (a) CA backward kernel
@pytest.mark.parametrize("n", [1, 3])
@pytest.mark.parametrize("h,w", [(1, 1), (13, 21), (113, 113)])
@pytest.mark.parametrize("cr", [4, 1])
def test_channel_attention_backward_matches_fp64_autograd(n, h, w, cr):
    """csr_channel_attention_backward against fp64 autograd of CALayer (rcan.py:50-68) times dout on the same bf16 operands.
    The skip gradient is not part of the kernel's output.  dres starts as NaN (every element must be written); the parameter
    accumulators start at 1 (they must be added to)."""
    from climsr_b200._lib import check, current_stream_ptr, lib
    c = 64
    g = torch.Generator().manual_seed(1000 * n + 10 * h + w + cr)
    res = _bf(torch.rand((n, c, h, w), generator=g) * 2 - 1)
    x = _bf(torch.rand((n, c, h, w), generator=g) * 2 - 1)
    dout = _bf(torch.rand((n, c, h, w), generator=g) * 2 - 1)
    w1 = (torch.rand((cr, c), generator=g) * 2 - 1) / 4
    b1 = torch.rand((cr,), generator=g) * 0.2 + 0.05         # hidden units alive ...
    if cr > 1:
        b1[0] = -8.0                                            # ... but one: its ReLU' = 0 must zero its gradients
    w2 = (torch.rand((c, cr), generator=g) * 2 - 1)
    b2 = torch.rand((c,), generator=g) - 0.5
    # reference
    p64 = [t.double().requires_grad_(True) for t in (res, w1, b1, w2, b2)]
    r64, W1, B1, W2, B2 = p64
    hid = F.relu(r64.mean(dim=(2, 3)) @ W1.t() + B1)
    gate = torch.sigmoid(hid @ W2.t() + B2)
    (r64 * gate[:, :, None, None] * dout.double()).sum().backward()
    # kernel: the forward leaves the pooled sums the backward reads
    rb, xb, db_ = _nhwc(res), _nhwc(x), _nhwc(dout)
    cw1, cb1, cw2, cb2 = (t.contiguous().cuda() for t in (w1, b1, w2, b2))
    out = torch.empty_like(rb)
    pooled = torch.empty((n, c), dtype=torch.float32, device="cuda")
    check(lib.csr_channel_attention(rb.data_ptr(), xb.data_ptr(), cw1.data_ptr(), cb1.data_ptr(), cw2.data_ptr(), cb2.data_ptr(), out.data_ptr(),
                                    pooled.data_ptr(), n, h, w, c, cr, current_stream_ptr()))
    dres = torch.full_like(rb, float("nan"))
    acc = [torch.ones_like(t) for t in (cw1, cb1, cw2, cb2)]
    nbytes = lib.csr_channel_attention_backward_scratch_bytes(n, c)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    check(lib.csr_channel_attention_backward(db_.data_ptr(), rb.data_ptr(), pooled.data_ptr(), cw1.data_ptr(), cb1.data_ptr(), cw2.data_ptr(),
                                             cb2.data_ptr(), dres.data_ptr(), acc[0].data_ptr(), acc[1].data_ptr(), acc[2].data_ptr(),
                                             acc[3].data_ptr(), scratch.data_ptr(), nbytes, n, h, w, c, cr, current_stream_ptr()))
    got = _nchw(dres, c)
    ref = r64.grad.float()
    assert torch.isfinite(got).all()
    assert float((got - ref).abs().max()) <= 2.0 ** -7 * float(ref.abs().max())
    for a, t in zip(acc, (W1, B1, W2, B2)):
        want = t.grad.double()
        err = float(((a.cpu().double() - 1) - want).abs().max())
        assert err <= 1e-3 * max(float(want.abs().max()), 1e-6), (err, float(want.abs().max()))
    if cr > 1:
        assert float((acc[1][0] - 1).abs()) == 0.0 and float((acc[0][0] - 1).abs().max()) == 0.0


# ---------------------------------------------------------------------------------------------------- (b) PixelUnshuffle
@pytest.mark.parametrize("n,h,w,c", [(1, 1, 1, 8), (2, 5, 7, 64), (3, 16, 16, 64), (1, 9, 4, 24)])
def test_pixel_unshuffle2_is_the_exact_adjoint_of_pixel_shuffle2(n, h, w, c):
    from climsr_b200._lib import check, current_stream_ptr, lib
    src = (torch.randn((n, 2 * h, 2 * w, c), generator=torch.Generator().manual_seed(h * w + c))).to(torch.bfloat16).cuda()
    dst = torch.full((n, h, w, 4 * c), float("nan"), dtype=torch.bfloat16, device="cuda")
    check(lib.csr_pixel_unshuffle2(src.data_ptr(), dst.data_ptr(), n, h, w, c, current_stream_ptr()))
    want = F.pixel_unshuffle(src.permute(0, 3, 1, 2), 2).permute(0, 2, 3, 1)
    assert torch.equal(dst, want)
    back = torch.empty_like(src)
    check(lib.csr_pixel_shuffle2(dst.data_ptr(), back.data_ptr(), n, h, w, c, current_stream_ptr()))
    assert torch.equal(back, src)


# ---------------------------------------------------------------------------------------------------- (c) conv shapes of the backward
def _conv_t_case(seed, n, h, w, cout_f, cin_f, k, gated, in_c=64, fill=0.0):
    """Input gradient of a forward conv (cout_f, cin_f, k, k) against fp64 conv_transpose2d on the bf16 operands, optionally
    times ReLU'(saved activation)."""
    from climsr_b200 import ops
    g = torch.Generator().manual_seed(seed)
    wt = (torch.rand((cout_f, cin_f, k, k), generator=g) * 2 - 1) / (cout_f * k * k) ** 0.5
    gy = _bf(torch.rand((n, cout_f, h, w), generator=g) * 2 - 1)
    want = F.conv_transpose2d(gy.double(), _bf(wt).double(), padding=k // 2).float()
    gate = None
    if gated:
        act = _bf(torch.rand((n, cin_f, h, w), generator=g) * 2 - 1)
        want = want * (act > 0).float()
        gate = _nhwc(act, (cin_f + 63) // 64 * 64)
    out = ops.conv2d_nhwc(_nhwc(gy, in_c, fill), wt.cuda(), None, transposed=True, gate=gate, gate_neg=0.0)
    got = _nchw(out, cin_f)
    assert torch.isfinite(got).all()
    assert float((got - want).abs().max()) <= 2.0 ** -7 * float(want.abs().max())


@pytest.mark.parametrize("n,h,w,cout_f,cin_f,k,gated,in_c,fill", [
    (2, 13, 21, 64, 64, 3, True, 64, 0.0),        # RCAB body.2: ReLU-gated (gate_neg = 0) 3x3 64 -> 64
    (2, 20, 24, 64, 64, 3, False, 64, 0.0),       # RCAB body.0 / group and body convs
    (2, 10, 12, 256, 64, 3, False, 256, 0.0),     # upsampler conv 64 -> 256
    (1, 40, 48, 1, 64, 3, False, 64, 9.0),        # tail.1 from the 1-channel gradient (channels >= 1 never multiplied)
    (1, 40, 48, 64, 3, 9, False, 64, 0.0),        # srcnn.conv1 9x9
    (1, 40, 48, 1, 32, 5, True, 64, 9.0),         # srcnn.conv3 5x5, gated by srcnn.conv2's ReLU
    (1, 40, 48, 32, 64, 1, True, 64, 0.0),        # srcnn.conv2 1x1, gated by srcnn.conv1's ReLU
])
def test_rcan_input_gradient_conv_shapes(n, h, w, cout_f, cin_f, k, gated, in_c, fill):
    _conv_t_case(h * w + k + cout_f, n, h, w, cout_f, cin_f, k, gated, in_c, fill)


def test_rcan_input_gradient_conv_with_two_residuals():
    """RCAB body.0's input gradient at the first block of a group: conv_t + RCAB skip (res1) + ResidualGroup skip (res2)."""
    from climsr_b200 import ops
    g = torch.Generator().manual_seed(3)
    n, h, w = 2, 13, 21
    wt = (torch.rand((64, 64, 3, 3), generator=g) * 2 - 1) / 24
    gy, r1, r2 = (_bf(torch.rand((n, 64, h, w), generator=g) * 2 - 1) for _ in range(3))
    want = F.conv_transpose2d(gy.double(), _bf(wt).double(), padding=1).float() + r1 + r2
    out = ops.conv2d_nhwc(_nhwc(gy), wt.cuda(), None, transposed=True, res1=_nhwc(r1), res2=_nhwc(r2))
    assert float((_nchw(out, 64) - want).abs().max()) <= 2.0 ** -7 * float(want.abs().max())


@pytest.mark.parametrize("n,h,w,cout,cin,k", [
    (2, 10, 12, 256, 64, 3),            # upsampler conv 64 -> 256 (job mode)
    (1, 33, 45, 256, 64, 3),
    (1, 40, 48, 64, 3, 9),              # srcnn.conv1 9x9: two output-channel chunks (9 x 64 accumulator columns exceed TMEM)
])
def test_rcan_wgrad_shapes(n, h, w, cout, cin, k):
    """Weight / bias gradients of the layer shapes only RCAN's backward has, accumulated onto ones."""
    from climsr_b200 import ops
    g = torch.Generator().manual_seed(n + h + w + k)
    x = _bf(torch.rand((n, cin, h, w), generator=g) * 2 - 1)
    gy = _bf(torch.rand((n, cout, h, w), generator=g) * 2 - 1)
    wt = torch.zeros((cout, cin, k, k), dtype=torch.float64, requires_grad=True)
    (dw_ref,) = torch.autograd.grad(F.conv2d(x.double(), wt, None, padding=k // 2), wt, gy.double())
    db_ref = gy.double().sum(dim=(0, 2, 3))
    dw = torch.ones((cout, cin, k, k), device="cuda")
    db = torch.ones((cout,), device="cuda")
    ops.conv2d_wgrad(_nhwc(x), _nhwc(gy, (cout + 63) // 64 * 64), (cout, cin, k, k), dw=dw, db=db)
    ew = float(((dw.cpu().double() - 1) - dw_ref).abs().max()) / max(1.0, float(dw_ref.abs().max()))
    eb = float(((db.cpu().double() - 1) - db_ref).abs().max()) / max(1.0, float(db_ref.abs().max()))
    assert ew <= 1e-3 and eb <= 1e-3, (ew, eb)


# ---------------------------------------------------------------------------------------------------- (d) reference golden
def _train_grads(net, x, elev, mask, wsum):
    net = net.cuda().train()
    net.zero_grad(set_to_none=True)
    sr = net(x.cuda(), elev.cuda(), mask.cuda())
    (sr * wsum.cuda()).sum().backward()
    return sr.detach().cpu(), {k: p.grad.detach().cpu() for k, p in net.named_parameters()}


def _is_ca(name):
    return ".conv_du." in name


def test_rcan_backward_matches_reference_golden(golden_dir):
    """tests/golden/rcan_grad.npz: gradients of the UNMODIFIED reference module (seed 0, 2 groups x 3 blocks, n = 2, LR 20 x 24,
    loss = sum(sr * w)).  Every parameter's sum |g| within GABS_CONV (convs) / GABS_CA (CALayer 1x1 convs), the four stored full
    tensors at cosine >= 0.99 and relative L2 <= FULL_REL.  Measured worsts on an NVIDIA B200 (1000 W): sum |g| 3.4 % (tail.1.bias)
    for the convs, 11.6 % for the CALayer convs; full tensors rel L2 5.2 % (tail.0.2.weight), cosine 0.9987."""
    from oracle import synth
    z = np.load(os.path.join(golden_dir, "rcan_grad.npz"))
    ng, nbk, n, h, w, seed = (int(v) for v in z["meta"])
    net = _rcan(ng, nbk, seed)
    x, elev, mask = synth.make_inputs(n, 3, h, w, seed=50 + seed)
    wsum = torch.randn((n, 1, 4 * h, 4 * w), generator=torch.Generator().manual_seed(77))
    _, grads = _train_grads(net, x, elev, mask, wsum)
    names = [str(k) for k in z["names"]]
    assert names == list(grads.keys())
    errs = {}
    for i, k in enumerate(names):
        assert torch.isfinite(grads[k]).all(), k
        ref = float(z["g_abs"][i])
        errs[k] = abs(float(grads[k].double().abs().sum()) - ref) / max(ref, 1e-12)
    full = {key[2:]: _metrics(grads[key[2:]], torch.from_numpy(z[key])) for key in z.files if key.startswith("g:")}
    print("golden: worst g_abs conv", max((v, k) for k, v in errs.items() if not _is_ca(k)),
          "CA", max((v, k) for k, v in errs.items() if _is_ca(k)), "full", full)
    for k, e in errs.items():
        assert e <= (GABS_CA if _is_ca(k) else GABS_CONV), (k, e)
    for k, (rel, cos) in full.items():
        assert cos >= 0.99 and rel <= FULL_REL, (k, rel, cos)


GABS_CONV, GABS_CA, FULL_REL = 0.07, 0.25, 0.1


# ---------------------------------------------------------------------------------------------------- (e) fp32 oracle, every parameter
def _oracle_grads(net, x, elev, mask, wsum, ng, nbk):
    from oracle import rcan as orc
    sd = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in net.state_dict().items()}
    (orc.rcan_forward(sd, x, elev, mask, ng, nbk) * wsum).sum().backward()
    return {k: v.grad for k, v in sd.items()}


# (ng, nbk): conv weight (rel L2, cosine), conv bias (rel L2, cosine), CALayer per-kind aggregate (rel L2, cosine).
# Measured worsts on an NVIDIA B200 (1000 W): 2 x 3 - conv tensors rel L2 7.7 % (a bias), cosine 0.9971; CALayer aggregates
# rel L2 7.8 %, cosine 0.9984.  10 x 20 - conv weights rel L2 17 %, cosine 0.985; conv biases rel L2 37 % (tail.1.bias, one
# cancelling scalar; rounding the reference's weights to bf16 alone moves it by 22 %), cosine 0.976; CALayer aggregates rel L2
# 12.2 %, cosine 0.9925.
ORACLE_BOUNDS = {
    (2, 3): ((0.15, 0.994), (0.15, 0.994), (0.15, 0.996)),
    (10, 20): ((0.35, 0.97), (0.75, 0.95), (0.25, 0.985)),
}


@pytest.mark.parametrize("ng,nbk,n,h,w", [(2, 3, 2, 20, 24), (10, 20, 2, 16, 16)])
def test_rcan_backward_matches_fp32_oracle_every_parameter(ng, nbk, n, h, w):
    """Every parameter's gradient against fp32 autograd of oracle/rcan.py with the same weights, at the golden's size and at the
    Hydra depth (10 groups x 20 blocks, conf/generator/rcan.yaml).

    Every conv weight and bias is held per tensor.  The CALayer 1x1 convs are held per kind (all blocks' conv_du.0.weight
    together, and so on): their gradients are products of two cancelling sums (over pixels, then over channels), and the fp32
    reference itself is not stable there - rounding only its conv weights to bf16 moves single CALayer gradients by a relative
    L2 of up to 11 at the Hydra depth (seed 3), while the per-kind aggregates move by <= 9 %.  The per-block kernel is held to
    1e-3 by test_channel_attention_backward_matches_fp64_autograd.  Measured worsts on a B200: next to ORACLE_BOUNDS."""
    from oracle import synth
    net = _rcan(ng, nbk, 3)
    x, elev, mask = synth.make_inputs(n, 3, h, w, seed=4)
    wsum = torch.randn((n, 1, 4 * h, 4 * w), generator=torch.Generator().manual_seed(5))
    _, grads = _train_grads(net, x, elev, mask, wsum)
    ref = _oracle_grads(net, x, elev, mask, wsum, ng, nbk)
    conv = {}
    for k, r in ref.items():
        assert torch.isfinite(grads[k]).all(), k
        if not _is_ca(k):
            conv[k] = _metrics(grads[k], r)
    agg = {}
    for kind in ("conv_du.0.weight", "conv_du.0.bias", "conv_du.2.weight", "conv_du.2.bias"):
        ks = [k for k in ref if k.endswith(kind)]
        agg[kind] = _metrics(torch.cat([grads[k].flatten() for k in ks]), torch.cat([ref[k].flatten() for k in ks]))
    for kind in ("weight", "bias"):
        sel = {k: v for k, v in conv.items() if k.endswith(kind)}
        print(f"oracle {ng}x{nbk} conv {kind}: worst rel", max((v[0], k) for k, v in sel.items()), "worst cos",
              min((v[1], k) for k, v in sel.items()))
    print(f"oracle {ng}x{nbk} CALayer aggregates", agg)
    (r_w, c_w), (r_b, c_b), (r_ca, c_ca) = ORACLE_BOUNDS[(ng, nbk)]
    for k, (rel, cos) in conv.items():
        bound = (r_w, c_w) if k.endswith("weight") else (r_b, c_b)
        assert rel <= bound[0] and cos >= bound[1], (k, rel, cos)
    for k, (rel, cos) in agg.items():
        assert rel <= r_ca and cos >= c_ca, (k, rel, cos)


# ---------------------------------------------------------------------------------------------------- (f) semantics
def _batch(n, h, w, seed):
    from oracle import synth
    x, elev, mask = synth.make_inputs(n, 3, h, w, seed=seed)
    hr = torch.rand((n, 1, 4 * h, 4 * w), generator=torch.Generator().manual_seed(seed + 9)) * 2 - 1
    return {"lr": x.cuda(), "hr": hr.cuda(), "elevation": elev.cuda(), "mask": mask.cuda()}


def test_rcan_pretraining_steps_then_inference_uses_the_updated_weights():
    """Three SuperResolutionTask(generator_type="rcan") pre-training steps with AdamW (pl_generator_pre_training.py:18-33): the
    loss stays finite and the weights move; the next eval forward equals the oracle on the updated state_dict."""
    from climsr_b200.task import SuperResolutionTask
    from oracle import rcan as orc
    net = _rcan(2, 3, 11).cuda()
    before = {k: v.detach().clone() for k, v in net.state_dict().items()}
    task = SuperResolutionTask(net, generator_type="rcan")
    opt = torch.optim.AdamW(net.parameters(), lr=1e-4)
    net.train()
    for step in range(3):
        batch = _batch(2, 12, 16, 20 + step)
        loss = task.training_step(batch, step)
        assert torch.isfinite(loss).all()
        opt.zero_grad(set_to_none=True)
        loss.backward()
        assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in net.parameters())
        opt.step()
    moved = [k for k, v in net.state_dict().items() if not torch.equal(v, before[k])]
    assert len(moved) == len(before)
    net.eval()
    batch = _batch(2, 12, 16, 40)
    with torch.no_grad():
        got = net(batch["lr"], batch["elevation"], batch["mask"]).cpu()
        sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}
        want = orc.rcan_forward(sd, batch["lr"].cpu(), batch["elevation"].cpu(), batch["mask"].cpu(), 2, 3)
    assert float((got - want).abs().max()) <= GEN_TOL


def test_rcan_two_forwards_then_two_backwards():
    """Each forward keeps its own saved activations: two forwards followed by their two backwards accumulate the sum of the
    gradients of the two run one at a time (to fp32-atomic summation noise)."""
    from oracle import synth
    net = _rcan(2, 2, 12).cuda().train()
    xs = [synth.make_inputs(2, 3, 16, 16, seed=s) for s in (1, 2)]
    ws = [torch.randn((2, 1, 64, 64), generator=torch.Generator().manual_seed(s)).cuda() for s in (3, 4)]
    outs = [net(x.cuda(), e.cuda(), m.cuda()) for x, e, m in xs]
    for o, wv in zip(outs, ws):
        (o * wv).sum().backward()
    both = {k: p.grad.clone() for k, p in net.named_parameters()}
    single = []
    for (x, e, m), wv in zip(xs, ws):
        net.zero_grad(set_to_none=True)
        (net(x.cuda(), e.cuda(), m.cuda()) * wv).sum().backward()
        single.append({k: p.grad.clone() for k, p in net.named_parameters()})
    for k, g in both.items():
        want = single[0][k] + single[1][k]
        assert float((g - want).abs().max()) <= 2e-5 * max(float(want.abs().max()), 1e-6), k


def test_rcan_refuses_input_gradients_and_frees_its_saved_activations():
    from climsr_b200 import CsrError
    from oracle import synth
    net = _rcan(1, 2, 13).cuda().train()
    x, e, m = (t.cuda() for t in synth.make_inputs(2, 3, 16, 16, seed=6))
    net(x, e, m).sum().backward()                       # warm-up: pack scratch, allocator pools
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    out = net(x, e, m)
    assert torch.cuda.memory_allocated() > base         # the node holds the saved activations ...
    del out
    torch.cuda.synchronize()
    assert torch.cuda.memory_allocated() == base        # ... and the graph releases them
    xg = x.clone().requires_grad_(True)
    with pytest.raises(CsrError):
        net(xg, e, m).sum().backward()
