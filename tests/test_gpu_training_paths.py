"""The generator training step as it actually runs, against a path or reference that is already tested.

test_gpu_backward.py compares the FIRST backward of a fresh plan, at most three RRDBs deep.  A training loop (and bench.py
--mode train) takes other paths: CUDA-graph capture and replay of the forward and backward on the plan's staging buffers, the
segmented backward of data-parallel training, the accumulate (+=) C entry point, the bf16 gradient wire format, reserved SMs
(option 30) and full depth (nb = 11, 23).  Each test here runs one of those paths and compares it with a tested one.

Bit-exactness.  The forward and the weight gradients are deterministic functions of their inputs as long as the weight-gradient
partial sums go through per-CTA slices plus a reduce (option 25 = 0, read when a plan is created), so launch-path comparisons
assert equality.  Bias gradients always end in fp32 atomics (bias_grad_kernel, bias_grad_planar_kernel) and are held to
2e-5 * max|ref|, as in test_atomic_and_deterministic_weight_gradient_accumulation_agree.
"""
import contextlib
import ctypes as C
import math

import pytest
import torch
import torch.nn.functional as F

from test_gpu_backward import _plan_masks

pytestmark = pytest.mark.gpu

CFG3 = (4, 11, 16)                         # in_channels, nb, gc of the Hydra generator bench.py --mode train times
OPTION_DEFAULTS = {11: 1, 12: 1 << 21, 25: 1, 30: 0}


@contextlib.contextmanager
def _options(settings):
    """Set csr options {key: value}; restore their defaults whatever happens."""
    from climsr_b200._lib import lib
    try:
        for k, v in settings.items():
            _set(k, v)
        yield
    finally:
        for k in settings:
            lib.csr_set_option(k, OPTION_DEFAULTS[k])


def _set(key, value):
    from climsr_b200._lib import check, lib
    check(lib.csr_set_option(key, int(value)), f"csr_set_option({key})")


def _net(sd, in_ch, nb, gc, train=True):
    from climsr_b200.models import ESRGANGenerator
    net = ESRGANGenerator(in_ch, 1, 64, nb, gc)
    net.load_state_dict(sd)
    return net.cuda().train(train)


def _inputs(n, in_ch, h, w, seed):
    from oracle import synth
    x, elev, mask = synth.make_inputs(n, in_ch, h, w, seed=seed)
    hr = torch.rand((n, 1, 4 * h, 4 * w), generator=torch.Generator().manual_seed(seed + 100)) * 2 - 1
    return x.cuda(), elev.cuda(), mask.cuda(), hr.cuda()


def _step(net, x, elev, mask, hr):
    """One training step through autograd: sr and every parameter gradient (fresh, not accumulated)."""
    net.zero_grad(set_to_none=True)
    sr = net(x, elev, mask)
    F.mse_loss(sr, hr).backward()
    return sr.detach().clone(), {k: p.grad.detach().clone() for k, p in net.named_parameters()}


def _train_plan(net, n, h, w):
    return net._plans[(n, h, w, next(net.parameters()).device, True)][0]


def _bias_close(got, ref, k=""):
    err = float((got - ref).abs().max())
    assert err <= 2e-5 * (float(ref.abs().max()) + 1e-12), (k, err)


def _assert_same_grads(got, ref):
    """Weight gradients bit for bit, bias gradients within the atomic-summation tolerance."""
    for k, r in ref.items():
        if k.endswith(".weight"):
            assert torch.equal(got[k], r), (k, float((got[k] - r).abs().max()))
        else:
            _bias_close(got[k], r, k)


def _oracle_errors(net, sd, x, elev, mask, hr, sr, grads, nb, gc):
    """max|sr - ref| and, per parameter, (rel L2, cosine, max|g - ref| / max|ref|) against the mask-matched fp32 oracle
    (test_gpu_backward.py): bf16-rounded weights and x, and the activation signs of the latest training forward of `net`."""
    from oracle import generator as og
    n, _, h, w = x.shape
    masks = _plan_masks(net, n, h, w, nb, gc)
    sd_q = {k: (v.to(torch.bfloat16).float() if k.endswith(".weight") else v) for k, v in sd.items()}
    x_q = x.cpu().to(torch.bfloat16).float()
    sr_ref, _, grads_ref = og.generator_forward_backward(sd_q, x_q, elev.cpu(), mask.cpu(), hr.cpu(), loss="mse", masks=masks)
    out = {}
    for k, ref in grads_ref.items():
        g = grads[k].cpu()
        assert torch.isfinite(g).all(), k
        rel = float((g - ref).norm() / (ref.norm() + 1e-30))
        cos = float(F.cosine_similarity(g.flatten().double(), ref.flatten().double(), dim=0))
        mx = float((g - ref).abs().max() / (ref.abs().max() + 1e-30))
        out[k] = (rel, cos, mx)
    return float((sr.cpu() - sr_ref).abs().max()), out


def _assert_mask_matched_bounds(sr_err, errs):
    """The bounds of test_generator_backward_matches_mask_matched_oracle."""
    assert sr_err <= 1e-2, sr_err
    for k, (rel, cos, _) in errs.items():
        if k.endswith(".weight"):
            assert rel <= 2e-2 and cos >= 0.9995, (k, rel, cos)
        else:
            assert rel <= 4e-2 and cos >= 0.999, (k, rel, cos)


def _perturb(nets, gen):
    """The same seeded, in-place relative change of every parameter of every net (no optimizer: its input, the bias gradients,
    is not bit-reproducible, so two nets stepped by it would drift apart)."""
    with torch.no_grad():
        for k, p in nets[0].named_parameters():
            f = (1 + 0.05 * (torch.rand(p.shape, generator=gen) * 2 - 1)).cuda()
            for net in nets:
                dict(net.named_parameters())[k].mul_(f)


# ---------------------------------------------------------------------------------------------------------- 1. graph replay
def test_graph_replayed_training_steps_match_direct_launches():
    """Four training steps with CUDA-graph replay (option 11 = 1: call 1 direct, call 2 captured, calls 3-4 replayed on the plan's
    staging buffers) against the same steps launched directly (option 11 = 0).  Inputs, targets and weights change before every
    step, so a replay that read a stale operand shows up.  cfg3 network at a batch under the option-12 pixel limit.  Every step is
    also held to the mask-matched fp32 oracle, which catches a fault both launch paths share (a dL/dout that never reaches the
    plan's staging buffer gives both the same zero gradients)."""
    from climsr_b200._lib import lib
    from oracle import synth
    in_ch, nb, gc = CFG3
    n, h, w = 2, 24, 20
    sd = synth.make_state_dict(in_ch, 1, 64, nb, gc, seed=31, gain=1.3)
    gen = torch.Generator().manual_seed(32)
    with _options({25: 0, 11: 1}):
        graphed, direct = _net(sd, in_ch, nb, gc), _net(sd, in_ch, nb, gc)
        for step in range(4):
            x, elev, mask, hr = _inputs(n, in_ch, h, w, seed=40 + step)
            _perturb([graphed, direct], gen)
            _set(11, 0)
            sr_d, g_d = _step(direct, x, elev, mask, hr)
            _set(11, 1)
            sr_g, g_g = _step(graphed, x, elev, mask, hr)
            assert torch.equal(sr_g, sr_d), step
            _assert_same_grads(g_g, g_d)
            plan_g, plan_d = _train_plan(graphed, n, h, w), _train_plan(direct, n, h, w)
            if step >= 2:
                assert lib.csr_plan_graph_status(plan_g, 0) == 1 and lib.csr_plan_graph_status(plan_g, 1) == 1, step
            assert lib.csr_plan_graph_status(plan_d, 0) == 0 and lib.csr_plan_graph_status(plan_d, 1) == 0
            # independent of both launch paths: a path both share (the dL/dout staging, say) is checked here
            sd_now = {k: v.detach().cpu() for k, v in graphed.state_dict().items()}
            _assert_mask_matched_bounds(*_oracle_errors(graphed, sd_now, x, elev, mask, hr, sr_g, g_g, nb, gc))


@pytest.mark.parametrize("replay", [True, False], ids=["replayed", "over_pixel_limit"])
def test_graph_replayed_inference_matches_direct_launches(replay):
    """Four eval forwards with new inputs each, the weights changed in place (plus mark_weights_dirty) before the fourth, against
    direct launches.  With option 12 below the plan's HR-pixel count the forward never enters the graph path.  Every call adds
    exactly csr_plan_num_launches to the launch counter, whether it launches directly, captures or replays."""
    from climsr_b200 import kernel_launch_count
    from climsr_b200._lib import lib
    from oracle import generator as og
    from oracle import synth
    in_ch, nb, gc = CFG3
    n, h, w = 2, 24, 20
    hr_px = n * 16 * h * w
    sd = synth.make_state_dict(in_ch, 1, 64, nb, gc, seed=33)
    gen = torch.Generator().manual_seed(34)
    with _options({11: 1, 12: OPTION_DEFAULTS[12] if replay else hr_px - 1}):
        graphed, direct = _net(sd, in_ch, nb, gc, train=False), _net(sd, in_ch, nb, gc, train=False)
        plan = graphed._plan(n, h, w, torch.device("cuda", torch.cuda.current_device()))
        with torch.no_grad():
            for call in range(4):
                x, elev, mask, _ = _inputs(n, in_ch, h, w, seed=50 + call)
                if call == 3:
                    _perturb([graphed, direct], gen)
                    graphed.mark_weights_dirty()
                    direct.mark_weights_dirty()
                graphed.packed_weights()
                l0 = kernel_launch_count()
                out_g = graphed(x, elev, mask)
                assert kernel_launch_count() - l0 == lib.csr_plan_num_launches(plan), call
                _set(11, 0)
                out_d = direct(x, elev, mask)
                _set(11, 1)
                assert torch.equal(out_g, out_d), call
                status = lib.csr_plan_graph_status(plan, 0)
                if not replay:
                    assert status == 0, call
                elif call >= 2:
                    assert status == 1, call
    want = og.generator_forward({k: v.detach().cpu() for k, v in graphed.state_dict().items()}, x.cpu(), elev.cpu(), mask.cpu())
    assert float((out_g.cpu() - want).abs().max()) <= 1e-2          # the changed weights were used


# ---------------------------------------------------------------------------------------------------- 2. segmented backward
def _flat_layout(net, plan):
    """(offset, numel, is_bias) of every gradient tensor inside the plan's flat buffer."""
    offs = net._grad_offsets(plan)
    params = [p for wb in net._ordered_params() for p in wb]
    return [(offs[i], p.numel(), i % 2 == 1) for i, p in enumerate(params)]


def _assert_same_flat(got, ref, layout):
    for off, k, is_bias in layout:
        g, r = got[off:off + k], ref[off:off + k]
        if is_bias:
            _bias_close(g, r, off)
        else:
            assert torch.equal(g, r), (off, float((g - r).abs().max()))


def test_segmented_backward_ranges_are_complete_and_match_flat_backward():
    """csr_plan_backward_segments / csr_plan_backward_flat_seg (the overlapped all-reduce path) against csr_plan_backward_flat on
    the same forward.  The flat buffer starts as NaN, so a range that is never copied stays NaN, and a range copied before its last
    writer ran differs from the unsegmented result.  Three runs per segmentation: direct, captured and replayed segment graphs."""
    from climsr_b200._lib import check, current_stream_ptr, lib
    from oracle import synth
    in_ch, nb, gc = CFG3
    n, h, w = 2, 24, 20
    sd = synth.make_state_dict(in_ch, 1, 64, nb, gc, seed=35, gain=1.3)
    x, elev, mask, _ = _inputs(n, in_ch, h, w, seed=60)
    go = (torch.rand((n, 1, 4 * h, 4 * w), generator=torch.Generator().manual_seed(61)) * 2 - 1).cuda() * 1e-3
    with _options({25: 0}):
        net = _net(sd, in_ch, nb, gc)
        net(x, elev, mask)                                    # training forward: the plan's saved activations
        plan = _train_plan(net, n, h, w)
        packed_bwd = net.packed_weights_bwd(force=True)
        nfl = lib.csr_plan_grad_floats(plan)
        layout = _flat_layout(net, plan)
        boundaries = {off for off, _, _ in layout} | {0, nfl}
        s = current_stream_ptr()
        ref = torch.empty(nfl, dtype=torch.float32, device="cuda")
        check(lib.csr_plan_backward_flat(plan, packed_bwd.data_ptr(), go.data_ptr(), ref.data_ptr(), s), "csr_plan_backward_flat")
        assert torch.isfinite(ref).all()
        lo, hi = C.c_size_t(), C.c_size_t()
        for nseg in (1, 2, 3, 8, 500):
            nk = lib.csr_plan_backward_segments(plan, nseg)
            assert 1 <= nk <= nseg, (nseg, nk)
            for run in range(3):
                flat = torch.full((nfl,), float("nan"), dtype=torch.float32, device="cuda")
                ranges = []
                for k in range(nk):
                    check(lib.csr_plan_backward_flat_seg(plan, packed_bwd.data_ptr(), go.data_ptr(), flat.data_ptr(), k, C.byref(lo),
                                                         C.byref(hi), s), "csr_plan_backward_flat_seg")
                    ranges.append((int(lo.value), int(hi.value)))
                assert ranges[0][1] == nfl and ranges[-1][0] == 0, (nseg, ranges)
                assert all(a <= b for a, b in ranges), (nseg, ranges)                              # empty ranges allowed
                assert all(r[0] == q[1] for r, q in zip(ranges, ranges[1:])), (nseg, ranges)       # contiguous, descending
                assert all(a in boundaries for a, _ in ranges), (nseg, ranges)
                assert not torch.isnan(flat).any(), (nseg, run, int(torch.isnan(flat).nonzero()[0]))
                _assert_same_flat(flat, ref, layout)
        again = torch.empty_like(ref)                          # the backward leaves the saved activations as they were
        check(lib.csr_plan_backward_flat(plan, packed_bwd.data_ptr(), go.data_ptr(), again.data_ptr(), s), "csr_plan_backward_flat")
        _assert_same_flat(again, ref, layout)


class _RecordingSync:
    """Stands in for parallel.BackwardGradSync with two ranks: records the slices the autograd node hands over, exchanges nothing."""
    world = 2
    nseg = 3

    def __init__(self):
        self.ranges = []

    def reduce_slice_async(self, flat, lo, hi, pending):
        self.ranges.append((lo, hi))

    def finish(self, flat, pending):
        pass


def test_autograd_segmented_backward_matches_unsegmented():
    """The `sync.world > 1` branch of GeneratorFunction.backward on one GPU: the gradients it returns equal those of the plain
    backward, and the slices it hands to the sync object tile the flat buffer from the top down."""
    from climsr_b200._lib import lib
    from oracle import synth
    in_ch, nb, gc = CFG3
    n, h, w = 2, 24, 20
    sd = synth.make_state_dict(in_ch, 1, 64, nb, gc, seed=36, gain=1.3)
    with _options({25: 0}):
        plain, seg = _net(sd, in_ch, nb, gc), _net(sd, in_ch, nb, gc)
        sync = _RecordingSync()
        seg.set_grad_sync(sync)
        for step in range(3):                                   # direct, captured and replayed segment graphs
            x, elev, mask, hr = _inputs(n, in_ch, h, w, seed=70 + step)
            sr_p, g_p = _step(plain, x, elev, mask, hr)
            sync.ranges = []
            sr_s, g_s = _step(seg, x, elev, mask, hr)
            assert torch.equal(sr_s, sr_p)
            _assert_same_grads(g_s, g_p)
            nfl = lib.csr_plan_grad_floats(_train_plan(seg, n, h, w))
            assert 1 <= len(sync.ranges) <= 3 and sync.ranges[0][1] == nfl and sync.ranges[-1][0] == 0, sync.ranges
            assert all(a[0] == b[1] for a, b in zip(sync.ranges, sync.ranges[1:])), sync.ranges


# ------------------------------------------------------------------------------------------------- 3. accumulate C entry point
def _grad_arrays(tensors):
    arr = (C.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = t.data_ptr() if t is not None else None
    return arr


def test_plan_backward_accumulates_into_caller_buffers():
    """csr_plan_backward (dw[i] += dL/dW_i, db[i] += dL/db_i into caller-owned buffers) against csr_plan_backward_flat on the same
    forward: from seeded D0, two calls give D0 + 2 * flat to fp32 rounding; from zero, one call gives the flat weights bit for bit.
    A null entry is refused with CSR_ERR_BAD_ARG before anything is launched or written."""
    from climsr_b200 import kernel_launch_count
    from climsr_b200._lib import check, current_stream_ptr, lib
    from oracle import synth
    in_ch, nb, gc = CFG3
    n, h, w = 2, 24, 20
    sd = synth.make_state_dict(in_ch, 1, 64, nb, gc, seed=37, gain=1.3)
    x, elev, mask, _ = _inputs(n, in_ch, h, w, seed=80)
    go = (torch.rand((n, 1, 4 * h, 4 * w), generator=torch.Generator().manual_seed(81)) * 2 - 1).cuda() * 1e-3
    with _options({25: 0}):
        net = _net(sd, in_ch, nb, gc)
        net(x, elev, mask)
        plan = _train_plan(net, n, h, w)
        pb = net.packed_weights_bwd(force=True).data_ptr()
        s = current_stream_ptr()
        pairs = net._ordered_params()
        offs = net._grad_offsets(plan)
        flat = torch.empty(lib.csr_plan_grad_floats(plan), dtype=torch.float32, device="cuda")
        check(lib.csr_plan_backward_flat(plan, pb, go.data_ptr(), flat.data_ptr(), s), "csr_plan_backward_flat")
        ref = [flat[offs[i]:offs[i] + p.numel()].view(p.shape) for i, p in enumerate(q for wb in pairs for q in wb)]

        g = torch.Generator().manual_seed(82)
        d0 = [((torch.rand(r.shape, generator=g) * 2 - 1) * float(r.abs().max() + 1e-3)).cuda() for r in ref]
        acc = [t.clone() for t in d0]
        dw, db = _grad_arrays(acc[0::2]), _grad_arrays(acc[1::2])
        for _ in range(2):
            check(lib.csr_plan_backward(plan, pb, go.data_ptr(), dw, db, s), "csr_plan_backward")
        for i, (a, d, r) in enumerate(zip(acc, d0, ref)):
            want = d + 2 * r
            tol = 1e-6 * float((d.abs() + 2 * r.abs()).max())
            if i % 2:
                tol += 2 * 2e-5 * (float(r.abs().max()) + 1e-12)
            assert float((a - want).abs().max()) <= tol, (i, float((a - want).abs().max()), tol)

        zero = [torch.zeros_like(r) for r in ref]
        check(lib.csr_plan_backward(plan, pb, go.data_ptr(), _grad_arrays(zero[0::2]), _grad_arrays(zero[1::2]), s), "csr_plan_backward")
        for i, (z, r) in enumerate(zip(zero, ref)):
            if i % 2:
                _bias_close(z, r, i)
            else:
                assert torch.equal(z, r), i

        nl = len(pairs)
        for which, layer in (("dw", 0), ("dw", nl // 2), ("dw", nl - 1), ("db", 1), ("db", nl - 2), ("db", nl - 1)):
            before = [t.clone() for t in acc]
            ws, bs = list(acc[0::2]), list(acc[1::2])
            (ws if which == "dw" else bs)[layer] = None
            torch.cuda.synchronize()
            l0 = kernel_launch_count()
            rc = lib.csr_plan_backward(plan, pb, go.data_ptr(), _grad_arrays(ws), _grad_arrays(bs), s)
            torch.cuda.synchronize()
            assert rc == -1, (which, layer, rc)                                        # CSR_ERR_BAD_ARG
            msg = lib.csr_last_error().decode()
            assert ("null weight-gradient pointer" if which == "dw" else "null bias-gradient pointer") in msg, msg
            assert kernel_launch_count() == l0, (which, layer)
            assert all(torch.equal(a, b) for a, b in zip(acc, before)), (which, layer)


# ------------------------------------------------------------------------------------------------------------ 4. full depth
# Bounds (max|sr - ref|; weights: rel L2, cosine, normalised max; biases: the same three), each about twice the worst tensor
# measured on an NVIDIA B200 (1000 W power limit):
#   nb = 11: sr 0.0020; weights rel 0.97 %, 1 - cos 4.5e-5, max 1.33 %; biases rel 0.98 %, 1 - cos 4.5e-5, max 1.42 %
#   nb = 23: sr 0.0144; weights rel 1.59 %, 1 - cos 1.2e-4, max 2.29 %; biases rel 1.46 %, 1 - cos 9.5e-5, max 1.82 %
# (nb <= 3: 0.8 % / 1.1 %, test_generator_backward_matches_mask_matched_oracle).  A missing or mis-scaled term gives >= 0.2.
FULL_DEPTH = [
    # in_ch, nb, gc, n, h, w, sr bound, (weight rel, cos, max), (bias rel, cos, max)
    (4, 11, 16, 16, 32, 32, 1e-2, (2e-2, 0.9995, 3e-2), (3e-2, 0.9995, 3e-2)),
    (4, 23, 32, 1, 16, 16, 3e-2, (3e-2, 0.9995, 4.5e-2), (3e-2, 0.9995, 4e-2)),
]


@pytest.mark.parametrize("in_ch,nb,gc,n,h,w,sr_tol,wtol,btol", FULL_DEPTH, ids=["cfg3_train", "class_default"])
def test_full_depth_backward_matches_mask_matched_oracle(in_ch, nb, gc, n, h, w, sr_tol, wtol, btol):
    """(a) the op list bench.py --mode train times on one GPU: cfg3 (in=4, nb=11, gc=16) at batch 16, LR 32x32, default options
    (whatever dense-block backward option 31 picks at this size); (b) the class-default net (in=4, nb=23, gc=32).  Every
    parameter against the mask-matched fp32 oracle by relative L2, cosine and max|g - ref| / max|ref| (an error confined to a few
    rows of a tensor hides inside an L2 norm, not inside the max).  The forward drifts further from the fp32 oracle with depth
    (bf16 activations), hence the per-depth bound on sr."""
    from oracle import synth
    sd = synth.make_state_dict(in_ch, 1, 64, nb, gc, seed=5, gain=1.3)
    x, elev, mask, hr = _inputs(n, in_ch, h, w, seed=90)
    net = _net(sd, in_ch, nb, gc)
    sr, grads = _step(net, x, elev, mask, hr)
    sr_err, errs = _oracle_errors(net, sd, x, elev, mask, hr, sr, grads, nb, gc)
    assert sr_err <= sr_tol, sr_err
    for k, (rel, cos, mx) in errs.items():
        rel_tol, cos_tol, max_tol = wtol if k.endswith(".weight") else btol
        assert rel <= rel_tol and cos >= cos_tol and mx <= max_tol, (k, rel, cos, mx)


# ---------------------------------------------------------------------------------------------------------- 5. reserved SMs
def test_reserved_sms_change_scheduling_only():
    """Option 30 = 4 (the attach_ddp default) shrinks every persistent grid and the number of weight-gradient partial slices of
    the plans created after it.  cfg3 at batch 16, LR 32x32: the forward is bit-identical, the weight gradients differ only by
    the summation order of the slices."""
    from oracle import synth
    in_ch, nb, gc = CFG3
    n, h, w = 16, 32, 32
    sd = synth.make_state_dict(in_ch, 1, 64, nb, gc, seed=38, gain=1.3)
    x, elev, mask, hr = _inputs(n, in_ch, h, w, seed=95)
    with _options({25: 0, 30: 4}):
        reserved = _net(sd, in_ch, nb, gc)
        sr_r, g_r = _step(reserved, x, elev, mask, hr)
        _set(30, 0)
        full = _net(sd, in_ch, nb, gc)
        sr_f, g_f = _step(full, x, elev, mask, hr)
    assert torch.equal(sr_r, sr_f)
    for k, ref in g_f.items():
        _bias_close(g_r[k], ref, k)


# ------------------------------------------------------------------------------------------------ 6. gradient wire format
def _wire_values(n, seed):
    """fp32 values with the edge cases of a bf16 conversion at the front: signed zeros, denormals, round-half-even ties, values
    that round up to bf16 infinity (at scale 1), infinities and NaN; seeded normals over many magnitudes behind them."""
    special = torch.tensor([0.0, -0.0, 1e-40, -1e-40, 1.4e-45, -3e-39, 1 + 2 ** -8, 1 + 3 * 2 ** -8, -(1 + 2 ** -8),
                            3.4e38, -3.4e38, 3.3895e38, math.inf, -math.inf, math.nan, 6.5e-38], dtype=torch.float32)
    g = torch.Generator().manual_seed(seed)
    body = torch.randn(n, generator=g) * torch.pow(10.0, torch.randint(-30, 30, (n,), generator=g).float())
    body[:min(n, special.numel())] = special[:n]
    return body


def _same_bits(got, want):
    nan_g, nan_w = torch.isnan(got), torch.isnan(want)
    assert torch.equal(nan_g, nan_w)
    ib = torch.int16 if got.dtype == torch.bfloat16 else torch.int32
    a, b = got.view(ib), want.view(ib)
    bad = (a != b) & ~nan_w
    assert not bad.any(), (int(bad.sum()), got[bad][:4], want[bad][:4])


@pytest.mark.parametrize("scale", [1.0, 0.5, 0.125])
@pytest.mark.parametrize("n", [0, 1, 7, 513, (1 << 20) + 3])
@pytest.mark.parametrize("lo", [0, 3])
def test_grad_wire_format_kernels_match_torch(scale, n, lo):
    """csr_grad_pack_bf16 == (flat * scale).to(bfloat16) and csr_grad_unpack_bf16 == comm.float() * scale, bit for bit (NaN stays
    NaN), computed on the host.  `lo` starts the slice off a 16-byte boundary as reduce_slice_async does (flat.data_ptr() + 4 * lo);
    n above 1024 runs the grid-stride loop (2 blocks of 512 threads); the elements around the slice are never touched."""
    from climsr_b200 import kernel_launch_count
    from climsr_b200._lib import check, current_stream_ptr, lib
    guard = 5
    src = _wire_values(n, seed=n + 7)
    flat = torch.full((lo + n + guard,), 7.0, dtype=torch.float32)
    flat[lo:lo + n] = src
    flat_d = flat.cuda()
    comm_d = torch.full((lo + n + guard,), -3.0, dtype=torch.bfloat16, device="cuda")
    s = current_stream_ptr()
    l0 = kernel_launch_count()
    check(lib.csr_grad_pack_bf16(flat_d.data_ptr() + 4 * lo, comm_d.data_ptr() + 2 * lo, n, scale, s), "csr_grad_pack_bf16")
    comm = comm_d.cpu()
    _same_bits(comm[lo:lo + n], (src * scale).to(torch.bfloat16))
    assert torch.equal(comm[:lo], torch.full((lo,), -3.0, dtype=torch.bfloat16))
    assert torch.equal(comm[lo + n:], torch.full((guard,), -3.0, dtype=torch.bfloat16))

    wire = src.to(torch.bfloat16)
    comm_d[lo:lo + n] = wire.cuda()
    out_d = torch.full((lo + n + guard,), 11.0, dtype=torch.float32, device="cuda")
    check(lib.csr_grad_unpack_bf16(comm_d.data_ptr() + 2 * lo, out_d.data_ptr() + 4 * lo, n, scale, s), "csr_grad_unpack_bf16")
    out = out_d.cpu()
    _same_bits(out[lo:lo + n], wire.float() * scale)
    assert torch.equal(out[:lo], torch.full((lo,), 11.0)) and torch.equal(out[lo + n:], torch.full((guard,), 11.0))
    assert kernel_launch_count() - l0 == (2 if n else 0)


# ------------------------------------------------------------------------------------------------ 7. caller-captured calls
@pytest.mark.parametrize("mode", ["global", "thread_local"])
def test_forward_and_backward_captured_by_the_caller(mode):
    """csr_plan_forward and csr_plan_backward_flat inside the caller's torch.cuda.graph capture (after one warm-up call each):
    the launches go into the caller's graph, the plan starts no capture of its own, and two replays with new inputs copied into
    the static tensors equal direct launches bit for bit (bias gradients: atomic tolerance).  Afterwards the plan's own graph
    path still captures and replays."""
    from climsr_b200._lib import check, current_stream_ptr, lib
    from oracle import synth
    in_ch, nb, gc = CFG3
    n, h, w = 2, 24, 20
    sd = synth.make_state_dict(in_ch, 1, 64, nb, gc, seed=39, gain=1.3)
    with _options({25: 0, 11: 1}):
        net = _net(sd, in_ch, nb, gc)
        x, elev, mask, _ = _inputs(n, in_ch, h, w, seed=100)
        net(x, elev, mask)                                     # creates the training plan; call 1 of its forward
        plan = _train_plan(net, n, h, w)
        layout = _flat_layout(net, plan)
        pf = net.packed_weights(force=True).data_ptr()
        pb = net.packed_weights_bwd(force=True).data_ptr()
        nfl = lib.csr_plan_grad_floats(plan)
        sx, se, sm = x.clone(), elev.clone(), mask.clone()
        sout = torch.empty((n, 1, 4 * h, 4 * w), dtype=torch.float32, device="cuda")
        sgo = torch.zeros_like(sout)
        sflat = torch.empty(nfl, dtype=torch.float32, device="cuda")

        def fwd(xx, ee, mm, out):
            check(lib.csr_plan_forward(plan, pf, xx.data_ptr(), ee.data_ptr(), mm.data_ptr(), out.data_ptr(), current_stream_ptr()),
                  "csr_plan_forward")

        def bwd(go, flat):
            check(lib.csr_plan_backward_flat(plan, pb, go.data_ptr(), flat.data_ptr(), current_stream_ptr()), "csr_plan_backward_flat")

        bwd(sgo, sflat)                                        # warm-up: call 1 of the backward
        torch.cuda.synchronize()
        gf, gb = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        with torch.cuda.graph(gf, capture_error_mode=mode):
            fwd(sx, se, sm, sout)
        with torch.cuda.graph(gb, capture_error_mode=mode):
            bwd(sgo, sflat)
        assert lib.csr_plan_graph_status(plan, 0) == 0 and lib.csr_plan_graph_status(plan, 1) == 0

        def direct(xx, ee, mm, go):
            out, flat = torch.empty_like(sout), torch.empty_like(sflat)
            _set(11, 0)
            try:
                fwd(xx, ee, mm, out)
                bwd(go, flat)
            finally:
                _set(11, 1)
            return out, flat

        for rep in range(2):
            x, elev, mask, _ = _inputs(n, in_ch, h, w, seed=101 + rep)
            go = (torch.rand(sout.shape, generator=torch.Generator().manual_seed(110 + rep)) * 2 - 1).cuda() * 1e-3
            sx.copy_(x), se.copy_(elev), sm.copy_(mask), sgo.copy_(go)
            gf.replay()
            gb.replay()
            got_out, got_flat = sout.clone(), sflat.clone()
            want_out, want_flat = direct(x, elev, mask, go)
            assert torch.equal(got_out, want_out), rep
            _assert_same_flat(got_flat, want_flat, layout)
        for call in range(2):                                  # the plan's own graphs: capture, then replay
            out, flat = torch.empty_like(sout), torch.empty_like(sflat)
            fwd(x, elev, mask, out)
            bwd(go, flat)
            assert torch.equal(out, want_out), call
            _assert_same_flat(flat, want_flat, layout)
        assert lib.csr_plan_graph_status(plan, 0) == 1 and lib.csr_plan_graph_status(plan, 1) == 1
        del gf, gb
