"""GPU parity of the generator training step (SURVEY.md section 8a row a6): weight-gradient GEMM, input-gradient convs and
the whole csr_plan_backward chain against fp32 autograd of the oracle / golden gradients of the reference module.

Tolerance.  Activations and gradient maps are stored in bf16 (fp32 accumulate).  Running the UNMODIFIED reference fully
in bf16 (oracle calibration, DESIGN.md section 5) reproduces its own fp32 gradients only to a relative L2 error of
0.6 % (srcnn.conv3) ... 2.5 % (conv_last, srcnn.conv1) ... 9 % (first RDB), cosine >= 0.995; this path is held to the
same envelope: cosine >= 0.99 and relative L2 <= 0.15 for every parameter, <= 0.06 for the weights of the four layers
nearest the loss.
Single kernels are held to bf16 rounding of their own operands (exact operands -> <= 1e-3 relative).
"""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

WGRAD_CASES = [
    # n, h, w, cin, cout, k, up2
    (1, 8, 14, 64, 16, 1, 0),
    (1, 8, 14, 128, 64, 1, 0),
    (1, 8, 14, 64, 16, 3, 0),           # RDB conv1
    (2, 16, 16, 80, 16, 3, 0),          # RDB conv2
    (2, 33, 45, 128, 64, 3, 0),         # RDB conv5, ragged tiles
    (1, 20, 40, 32, 1, 5, 0),           # srcnn.conv3
    (1, 12, 20, 64, 64, 3, 1),          # upconv (nearest x2 on the input): four phase GEMMs scattered into 3x3
    (1, 24, 24, 192, 64, 3, 0),         # gc=32 conv5: two 128-channel chunks
    (1, 1, 1, 64, 64, 3, 0),            # single pixel
    (1, 113, 113, 64, 64, 3, 0),        # Europe-extent LR raster
    # the discriminator's ten convs at the GAN step's batch 16 (same-convs over the padded maps; job mode from 128 channels on)
    (16, 130, 130, 1, 64, 3, 0),        # stage 1 conv_a: one input channel in a 64-channel buffer
    (16, 130, 130, 64, 64, 3, 0),       # stage 1 conv_b
    (16, 66, 66, 64, 128, 3, 0),        # stage 2 conv_a
    (16, 66, 66, 128, 128, 3, 0),       # stage 2 conv_b
    (16, 34, 34, 128, 256, 3, 0),       # stage 3 conv_a
    (16, 34, 34, 256, 256, 3, 0),       # stage 3 conv_b
    (16, 18, 18, 256, 512, 3, 0),       # stage 4 conv_a
    (16, 18, 18, 512, 512, 3, 0),       # stage 4 conv_b
    (16, 8, 8, 512, 512, 3, 0),         # conv4
    (16, 6, 6, 512, 512, 3, 0),         # conv5
]


@pytest.mark.parametrize("n,h,w,cin,cout,k,up2", WGRAD_CASES)
def test_wgrad_matches_autograd(n, h, w, cin, cout, k, up2):
    from climsr_b200 import ops
    g = torch.Generator().manual_seed(n * 100 + h + cin + k)
    x = (torch.rand((n, cin, h, w), generator=g) * 2 - 1).to(torch.bfloat16).float()
    s = 2 if up2 else 1
    gy = (torch.rand((n, cout, s * h, s * w), generator=g) * 2 - 1).to(torch.bfloat16).float()
    wt = torch.zeros((cout, cin, k, k), dtype=torch.float64, requires_grad=True)
    xin = F.interpolate(x, scale_factor=2, mode="nearest") if up2 else x
    # fp64 on the GPU for the large layers (the same fp64 arithmetic, seconds instead of minutes on the host)
    dev = "cuda" if n * h * w * cin * cout > 1 << 26 else "cpu"
    wt = wt.detach().to(dev).requires_grad_(True)
    (dw_ref,) = torch.autograd.grad(F.conv2d(xin.to(dev).double(), wt, None, padding=k // 2), wt, gy.to(dev).double())
    dw_ref = dw_ref.cpu()
    db_ref = gy.double().sum(dim=(0, 2, 3))
    xb = torch.zeros((n, h, w, (cin + 63) // 64 * 64), dtype=torch.bfloat16)
    xb[..., :cin] = x.permute(0, 2, 3, 1).to(torch.bfloat16)
    gb = torch.full((n, s * h, s * w, (cout + 63) // 64 * 64), 3.0, dtype=torch.bfloat16)      # channels >= cout must never be used
    gb[..., :cout] = gy.permute(0, 2, 3, 1).to(torch.bfloat16)
    dw = torch.ones((cout, cin, k, k), device="cuda")                        # accumulate semantics: dw += scale * grad
    db = torch.ones((cout,), device="cuda")
    ops.conv2d_wgrad(xb.cuda(), gb.cuda(), (cout, cin, k, k), in_up2=bool(up2), scale=0.5, dw=dw, db=db)
    ew = float(((dw.cpu().double() - 1) * 2 - dw_ref).abs().max()) / max(1.0, float(dw_ref.abs().max()))
    eb = float(((db.cpu().double() - 1) * 2 - db_ref).abs().max()) / max(1.0, float(db_ref.abs().max()))
    assert ew <= 1e-3 and eb <= 1e-3, (ew, eb)


def _train_step(sd, x, elev, mask, hr, in_ch, nb, gc, loss="mse"):
    from climsr_b200.models import ESRGANGenerator
    net = ESRGANGenerator(in_ch, 1, 64, nb, gc)
    net.load_state_dict(sd)
    net = net.cuda().train()
    sr = net(x.cuda(), elev.cuda(), mask.cuda())
    lv = F.mse_loss(sr, hr.cuda()) if loss == "mse" else F.l1_loss(sr, hr.cuda())
    lv.backward()
    return sr.detach().cpu(), float(lv.detach()), {k: p.grad.detach().cpu() for k, p in net.named_parameters()}, net


def _check_grads(got, want, near_loss=("srcnn.conv3", "srcnn.conv2", "srcnn.conv1", "conv_last")):
    for k, ref in want.items():
        g = got[k]
        assert torch.isfinite(g).all(), k
        rel = float((g - ref).norm() / (ref.norm() + 1e-30))
        cos = float(F.cosine_similarity(g.flatten().double(), ref.flatten().double(), dim=0))
        # bias gradients are short vectors (16..64 sums with heavy cancellation, conv_last.bias a single scalar): the bf16
        # reference itself moves them by several percent, so they get the looser bounds
        is_bias = k.endswith(".bias")
        assert cos >= (0.98 if is_bias else 0.99), (k, cos)
        tight = k.endswith(".weight") and k.rsplit(".", 1)[0] in near_loss
        assert rel <= (0.06 if tight else 0.2 if is_bias else 0.15), (k, rel)


@pytest.mark.parametrize("in_ch,nb,gc,n,h,w", [(2, 1, 16, 2, 16, 16), (4, 2, 16, 1, 20, 12), (3, 1, 32, 1, 12, 12)])
def test_generator_backward_matches_oracle(in_ch, nb, gc, n, h, w):
    """Hydra-style (gc=16: dense-block weight-gradient GEMM) and class-default-style (gc=32: per-layer GEMMs, 192-channel
    concat pitch) blocks, ragged rasters."""
    from oracle import generator as og
    from oracle import synth
    sd = synth.make_state_dict(in_ch, 1, 64, nb, gc, seed=5)
    x, elev, mask = synth.make_inputs(n, in_ch, h, w, seed=6)
    hr = torch.rand((n, 1, 4 * h, 4 * w), generator=torch.Generator().manual_seed(7)) * 2 - 1
    sr_ref, loss_ref, grads_ref = og.generator_forward_backward(sd, x, elev, mask, hr, loss="mse")
    sr, lv, grads, _ = _train_step(sd, x, elev, mask, hr, in_ch, nb, gc)
    assert float((sr - sr_ref).abs().max()) <= 1e-2
    assert abs(lv - float(loss_ref)) <= 1e-3 * max(1.0, float(loss_ref))
    _check_grads(grads, grads_ref)


def _plan_masks(net, n, h, w, nb, gc):
    """Activation patterns of the latest TRAINING forward of `net`, read from its plan's saved activations (csr_plan_buffer):
    layer name -> bool NCHW tensor (True where the stored bf16 activation is positive; LeakyReLU / ReLU preserve the sign)."""
    import ctypes as C
    from climsr_b200._lib import check, lib
    plan, ws = net._plans[(n, h, w, next(net.parameters()).device, True)]
    base = (ws.data_ptr() + 1023) // 1024 * 1024 - ws.data_ptr()
    off, dims = C.c_size_t(), (C.c_int32 * 4)()

    def view(kind, index):
        check(lib.csr_plan_buffer(plan, kind, index, C.byref(off), C.byref(dims)), "csr_plan_buffer")
        nn_, hh, ww, cc = (int(v) for v in dims)
        nbytes = nn_ * hh * ww * cc * 2
        return ws[base + off.value: base + off.value + nbytes].view(torch.bfloat16).view(nn_, hh, ww, cc)

    masks = {}
    for i in range(nb):
        for r in range(3):
            cat = view(0, 3 * i + r)
            for k in range(1, 5):
                sl = cat[..., 64 + (k - 1) * gc: 64 + k * gc]
                masks[f"RRDB_trunk.{i}.RDB{r + 1}.conv{k}"] = (sl.float() > 0).permute(0, 3, 1, 2).cpu()
    for name, kind, c in (("upconv1", 1, 64), ("upconv2", 2, 64), ("HRconv", 3, 64), ("srcnn.conv1", 4, 64), ("srcnn.conv2", 5, 32)):
        masks[name] = (view(kind, 0)[..., :c].float() > 0).permute(0, 3, 1, 2).cpu()
    return masks


@pytest.mark.parametrize("in_ch,nb,gc,n,h,w", [(4, 2, 16, 2, 24, 20), (3, 1, 32, 1, 12, 12), (4, 3, 16, 1, 32, 32)])
def test_generator_backward_matches_mask_matched_oracle(in_ch, nb, gc, n, h, w):
    """VERDICT r1 weak #3: the backward GRAPH held to a tight tolerance.  The fp32 oracle is run with (a) the bf16-rounded
    weights the kernels multiply with and (b) the LeakyReLU / ReLU activation patterns of OUR forward (read from the training
    plan's saved activations) - a bf16-emulating reference: what remains is rounding of the stored activations / gradient maps
    (bf16) and summation order.  Every weight gradient must then agree to a relative L2 error of 2e-2 with cosine >= 0.9995
    (the free-running comparison above needs 0.15 / 0.99 only because ~1 % of near-zero pre-activations flip their sign in bf16
    and LeakyReLU's derivative jumps there; a missing or mis-scaled term in the backward would show up here at >= 0.2)."""
    from oracle import generator as og
    from oracle import synth
    sd = synth.make_state_dict(in_ch, 1, 64, nb, gc, seed=5, gain=1.3)
    x, elev, mask = synth.make_inputs(n, in_ch, h, w, seed=6)
    hr = torch.rand((n, 1, 4 * h, 4 * w), generator=torch.Generator().manual_seed(7)) * 2 - 1
    sr, lv, grads, net = _train_step(sd, x, elev, mask, hr, in_ch, nb, gc)
    masks = _plan_masks(net, n, h, w, nb, gc)
    sd_q = {k: (v.to(torch.bfloat16).float() if k.endswith(".weight") else v) for k, v in sd.items()}
    x_q = x.to(torch.bfloat16).float()
    sr_ref, loss_ref, grads_ref = og.generator_forward_backward(sd_q, x_q, elev, mask, hr, loss="mse", masks=masks)
    assert float((sr - sr_ref).abs().max()) <= 1e-2
    worst = ("", 0.0)
    for k, ref in grads_ref.items():
        g = grads[k]
        rel = float((g - ref).norm() / (ref.norm() + 1e-30))
        cos = float(F.cosine_similarity(g.flatten().double(), ref.flatten().double(), dim=0))
        if rel > worst[1]:
            worst = (k, rel)
        if k.endswith(".weight"):
            assert rel <= 2e-2 and cos >= 0.9995, (k, rel, cos)   # measured worst: 0.8 %
        else:                                   # biases: short vectors of heavily cancelling sums (conv_last.bias is one scalar)
            assert rel <= 4e-2 and cos >= 0.999, (k, rel, cos)    # measured worst: 1.1 %
    print("worst gradient tensor", worst)


def test_generator_backward_matches_reference_golden(golden_dir):
    """Weights, inputs, targets and gradients all produced by the UNMODIFIED reference module (oracle/make_golden.py)."""
    z = np.load(os.path.join(golden_dir, "gen_tiny_refinit.npz"))
    sd = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd/")}
    x, elev, mask, hr = (torch.from_numpy(z[k]) for k in ("x", "elev", "mask", "hr_mse"))
    _, lv, grads, _ = _train_step(sd, x, elev, mask, hr, 2, 1, 16)
    assert abs(lv - float(z["loss_mse"])) <= 1e-3 * float(z["loss_mse"])
    want = {k[len("gradmse/"):]: torch.from_numpy(z[k]) for k in z.files if k.startswith("gradmse/")}
    assert len(want) >= 30
    _check_grads(grads, want)
    for name, norm in zip(z["gradmse_names"], z["gradmse_norms"]):
        assert abs(float(grads[str(name)].norm()) - float(norm)) <= 0.15 * float(norm), name


def test_training_step_semantics():
    """(1) gradients accumulate across backward calls like autograd's; (2) an optimizer step repacks the weights and changes
    the output; (3) a stale backward (another forward ran in between) is refused; (4) eval/no_grad takes the inference plan."""
    from climsr_b200 import CsrError
    from climsr_b200.models import ESRGANGenerator
    torch.manual_seed(0)
    net = ESRGANGenerator(3, 1, 64, 1, 16).cuda().train()
    g = torch.Generator().manual_seed(3)
    x = (torch.rand((2, 3, 12, 12), generator=g) * 2 - 1).cuda()
    elev = torch.rand((2, 1, 48, 48), generator=g).cuda()
    mask = (torch.rand((2, 1, 48, 48), generator=g) > 0.3).float().cuda()
    hr = (torch.rand((2, 1, 48, 48), generator=g) * 2 - 1).cuda()
    opt = torch.optim.AdamW(net.parameters(), lr=1e-3)
    out1 = net(x, elev, mask)
    F.l1_loss(out1, hr).backward()
    g1 = net.conv_last.weight.grad.clone()
    F.l1_loss(net(x, elev, mask), hr).backward()
    assert torch.allclose(net.conv_last.weight.grad, 2 * g1, rtol=1e-3, atol=1e-7)
    opt.step()
    out2 = net(x, elev, mask)
    assert not torch.equal(out1, out2)
    stale = net(x, elev, mask)
    _ = net(x, elev, mask)
    with pytest.raises(CsrError):
        stale.sum().backward()
    net.eval()
    with torch.no_grad():
        out3 = net(x, elev, mask)
    assert out3.requires_grad is False and torch.allclose(out3, out2.detach(), atol=1e-6)
    losses = []
    net.train()
    opt = torch.optim.AdamW(net.parameters(), lr=2e-4)
    for _ in range(12):
        opt.zero_grad()
        lv = F.l1_loss(net(x, elev, mask), hr)
        lv.backward()
        opt.step()
        losses.append(float(lv.detach()))
    assert losses[-1] < losses[0]                      # the step actually descends


@pytest.mark.parametrize("fused", [True, False])
def test_inference_after_optimizer_step_uses_the_updated_weights(fused):
    """VERDICT r1 weak #1: torch.optim.AdamW(fused=True).step() updates parameters WITHOUT bumping ``p._version``, the key of the
    inference pack cache.  Sequence of a Lightning epoch: training forward/backward, optimizer step, then validation in eval()
    / no_grad.  The eval forward must run on the updated weights: bit-identical to a forced repack and to a fresh module
    loaded from the updated state_dict, and within tolerance of the oracle on those weights."""
    from climsr_b200.models import ESRGANGenerator
    from oracle import generator as og
    torch.manual_seed(0)
    net = ESRGANGenerator(3, 1, 64, 1, 16).cuda().train()
    g = torch.Generator().manual_seed(3)
    x = (torch.rand((2, 3, 12, 12), generator=g) * 2 - 1).cuda()
    elev = torch.rand((2, 1, 48, 48), generator=g).cuda()
    mask = (torch.rand((2, 1, 48, 48), generator=g) > 0.3).float().cuda()
    hr = (torch.rand((2, 1, 48, 48), generator=g) * 2 - 1).cuda()
    opt = torch.optim.AdamW(net.parameters(), lr=5e-4, fused=fused)
    with torch.no_grad():
        before = net(x, elev, mask).clone()                       # fills the inference pack cache
    for step in range(2):
        opt.zero_grad()
        F.l1_loss(net(x, elev, mask), hr).backward()
        if step == 1:
            # GAN pattern (pl_gan.py:41-61): a frozen-generator forward between backward and the optimizer step
            for p in net.parameters():
                p.requires_grad_(False)
            with torch.no_grad():
                _ = net(x, elev, mask)
            for p in net.parameters():
                p.requires_grad_(True)
        opt.step()
    net.eval()
    with torch.no_grad():
        after = net(x, elev, mask).clone()
        net.packed_weights(force=True)
        forced = net(x, elev, mask).clone()
    assert not torch.equal(before, after)
    assert torch.equal(after, forced)
    fresh = ESRGANGenerator(3, 1, 64, 1, 16)
    fresh.load_state_dict({k: v.detach().cpu() for k, v in net.state_dict().items()})
    fresh = fresh.cuda().eval()
    with torch.no_grad():
        assert torch.equal(fresh(x, elev, mask), after)
        want = og.generator_forward({k: v.detach().cpu() for k, v in net.state_dict().items()}, x.cpu(), elev.cpu(), mask.cpu())
    assert float((after.cpu() - want).abs().max()) <= 1e-2
    # behind-autograd updates need the explicit mark
    with torch.no_grad():
        net.conv_last.bias.data.add_(0.5)
        net.mark_weights_dirty()
        moved = net(x, elev, mask)
    assert float((moved - after).abs().max()) > 1e-3


def test_plan_cache_eviction_never_frees_a_live_training_plan():
    """ADVICE r1: with four cached plans a fifth shape used to destroy every plan, the training plan of a live autograd node
    included.  Now the least recently used inference plan goes and the backward still runs (and matches an undisturbed one)."""
    import copy
    from climsr_b200.models import ESRGANGenerator
    torch.manual_seed(0)
    net = ESRGANGenerator(3, 1, 64, 1, 16).cuda().train()
    g = torch.Generator().manual_seed(5)
    mk = lambda n, h, w: ((torch.rand((n, 3, h, w), generator=g) * 2 - 1).cuda(), torch.rand((n, 1, 4 * h, 4 * w), generator=g).cuda(),  # noqa: E731
                          (torch.rand((n, 1, 4 * h, 4 * w), generator=g) > 0.3).float().cuda())
    x, elev, mask = mk(2, 12, 12)
    F.l1_loss(net(x, elev, mask), torch.zeros((2, 1, 48, 48), device="cuda")).backward()
    ref = {k: p.grad.clone() for k, p in net.named_parameters()}
    net.zero_grad()
    out = net(x, elev, mask)
    with torch.no_grad():
        for (n, h, w) in ((1, 8, 8), (1, 9, 9), (1, 10, 10), (1, 11, 11), (1, 12, 13), (1, 13, 12)):
            net(*mk(n, h, w))
    assert len(net._plans) <= 4
    F.l1_loss(out, torch.zeros((2, 1, 48, 48), device="cuda")).backward()
    for k, p in net.named_parameters():
        scale = float(ref[k].abs().max()) + 1e-12
        assert float((p.grad - ref[k]).abs().max()) <= 2e-5 * scale, k
    # deep copies (EMA / SWA shadows) own their plans
    twin = copy.deepcopy(net).eval()
    assert twin._plans == {} and twin._packed is None
    with torch.no_grad():
        a = twin(x, elev, mask)
        b = net.eval()(x, elev, mask)
    assert torch.equal(a, b)
    del twin


def test_atomic_and_deterministic_weight_gradient_accumulation_agree():
    """Option 25: weight-gradient partial sums through red.global.add.v4.f32 (default) against the deterministic per-CTA
    slices + tree reduce.  Same products, different summation order over CTAs: equal to fp32 rounding."""
    from climsr_b200._lib import lib
    from oracle import synth
    sd = synth.make_state_dict(4, 1, 64, 1, 16, seed=3)
    x, elev, mask = synth.make_inputs(2, 4, 24, 20, seed=4)
    hr = torch.rand((2, 1, 96, 80), generator=torch.Generator().manual_seed(5)) * 2 - 1
    grads = []
    try:
        for atomic in (1, 0, 0):
            lib.csr_set_option(25, atomic)
            grads.append(_train_step(sd, x, elev, mask, hr, 4, 1, 16)[2])
    finally:
        lib.csr_set_option(25, 1)
    for k in grads[0]:
        if k.endswith(".weight"):                 # (bias gradients always end in a few fp32 atomics per block)
            assert torch.equal(grads[1][k], grads[2][k]), k                  # the slice + reduce path is run-to-run deterministic
        scale = float(grads[1][k].abs().max()) + 1e-12
        assert float((grads[0][k] - grads[1][k]).abs().max()) <= 2e-5 * scale, k


def test_dense_block_backward_kernel_matches_per_layer_input_gradients():
    """The four gated input-gradient convs of a dense block as ONE dataflow launch (rdb_tc.cu, backward form; option 27, used
    when a block has at least option-31 windows per SM) against four per-layer launches: same tiles, MMA order and epilogue
    arithmetic, so with the deterministic weight-gradient accumulation (option 25 = 0) every gradient is bit-identical."""
    from climsr_b200._lib import lib
    from oracle import synth
    sd = synth.make_state_dict(4, 1, 64, 2, 16, seed=8, gain=1.3)
    x, elev, mask = synth.make_inputs(3, 4, 36, 28, seed=9)
    hr = torch.rand((3, 1, 144, 112), generator=torch.Generator().manual_seed(10)) * 2 - 1
    res = []
    try:
        lib.csr_set_option(25, 0)
        lib.csr_set_option(31, 0)
        for dense in (1, 0):
            lib.csr_set_option(27, dense)
            res.append(_train_step(sd, x, elev, mask, hr, 4, 2, 16))
    finally:
        lib.csr_set_option(25, 1)
        lib.csr_set_option(27, 1)
        lib.csr_set_option(31, 2)
    assert torch.equal(res[0][0], res[1][0])                       # sr
    for k in res[0][2]:
        if k.endswith(".weight"):
            assert torch.equal(res[0][2][k], res[1][2][k]), k
        else:
            assert float((res[0][2][k] - res[1][2][k]).abs().max()) <= 2e-5 * (float(res[1][2][k].abs().max()) + 1e-12), k
