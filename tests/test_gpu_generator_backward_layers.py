"""Every launch of the generator backward, read back from the plan's gradient buffers (csr_plan_buffer kinds 10..17) and its flat
gradient buffer, and held element by element to a float64 recomputation from the operands that launch read.

The backward runs one segment per point where its completed gradient suffix grows (csr_plan_backward_segments with one segment per
gradient float), so it stops right after each layer's last gradient op, and the gradient buffers are cloned at every stop.  bwd_build
(api.cu) leaves every operand of every op between two stops intact at one of those two stops:

  stop                      ops since the previous stop, operand (stop it is read at) -> result (stop)
  0  srcnn.conv3 done       gcol: bf16(dL/dout) -> gO (0);  dW/db srcnn.conv3: hrE, gO (0), db from dL/dout (fp32)
  1  srcnn.conv2 done       srcnn.conv3 cols: gO, gate relu'(hrE) -> gP[:32] (1);  dW/db srcnn.conv2: hrD, gP[:32] (1)
  2  srcnn.conv1 done       srcnn.conv2: gP[:32] (1), gate relu'(hrD) -> gQ (2);  dW/db srcnn.conv1: hrC (27-channel im2col), gQ (2)
  3  conv_last done         srcnn.conv1 (9x9 transposed): gQ (2) -> gT[:3] (3);  gcol: gT[0] -> gcolB (3);  dW/db conv_last: hrB, gT[0] (3)
  4  HRconv done            conv_last cols: gcolB (3), gate lrelu'(hrB) -> gP (4);  dW/db HRconv: hrA, gP (4)
  5  upconv2 done           HRconv: gP (4), gate lrelu'(hrA) -> gQ (5);  dW/db upconv2: nearest-x2(m1), gQ (5)
  6  upconv1 done           upconv2, four phases in place, the last gated by lrelu'(m1): gQ (5) -> gm1 (6);  dW/db upconv1: up(t0), gm1 (6)
  7  trunk_conv done        upconv1, four phases: gm1 (6) -> gt0 (7);  dW/db trunk_conv: trunk output, gt0 (7)
  8  first dense block      trunk_conv: gt0 (7) -> gcat[0][:64] (8);  then as every block below
  8+b dense block b done    (b > 0) the previous block's wide conv: its Gb (b-1) + g_y (b-1) [+ G = gcat[Pb][:64] (b-1) for an RDB1]
                            -> the next Gb[:64] (b);  (RDB3) kScale: gcat[Pb][:64] (b) -> bf16(0.2 G) = Gb[:64] (b);  the four gated
                            narrow convs g4..g1, each from [g_y | g4 .. g_s+1] of Gb (b), gate lrelu'(x_s);  dW/db conv1..conv5: the
                            block's forward concat, Gb (b), conv5 scaled by 0.2
  last  conv_first done     the last RDB1's wide conv (as above);  dW/db conv_first: bf16(x), gcat[Pb][:64] (last) + gt0 (last)

Gb = [g_y | g4 | g3 | g2 | g1] rotates through the three gradient concat buffers as bwd_build's Pb / Qb / Rb do.

References: the bf16 operands as stored, the weights as the backward pack rounds them, bf16(fp32(w) * wscale) (0.2 for conv5's
block of every dense-block input gradient), the upconv phases as 2x2 convs whose taps are bf16 of the fp32 sums of the 3x3 taps
mapped to them (pack_weight_body), and gates `stored activation > 0 ? 1 : neg` (gate8).  An input gradient is the vector-Jacobian
product of the layer's linear map in float64 (autograd over F.conv2d), then gate * (acc + residuals).

Bounds, per element:  input gradients |got - ref| <= ulp_bf16(ref) + 2^-12 A with A = gate (sum |w||g|) + |r1| + |r2|, plus one
bf16 ulp of each of the three stored and re-read phase partials for upconv2 / upconv1;  weight gradients 2^-12 sum |x||g| per entry
(sum |g| for a bias).  Measured on a B200 (1000 W power limit), worst error / bound over all cases: 0.485 for the input gradients
(conv_last's, the bf16 store of the fp32 accumulator: half an ulp), 0.474 for the four-phase upconv input gradients, 1e-3 for weight
and bias gradients (fp32 sums are far inside 2^-12; a dropped image, tap row or batch tail is not).

Sensitivity controls (reference side only, cases with controls): circular instead of zero padding must break the bound on the edge
rows and columns of every KxK input gradient and somewhere in every KxK weight gradient; one dropped tap of one input channel must
break it for every input gradient; the gate replaced by 1 for every gated one; and, at n > 1, leaving the last image out of a
layer's weight and bias gradients.
"""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F
from torch.nn.grad import conv2d_weight

from test_gpu_generator_layers import REL, PlanBuffers, _bf, _conv, _nchw, _options, _phase_weights, _run, _ulp
from test_gpu_training_paths import _assert_same_flat, _flat_layout

pytestmark = pytest.mark.gpu

GRAD_KINDS = {"gO": 10, "gcolB": 11, "gT": 12, "gP": 13, "gQ": 14, "gm1": 15, "gt0": 16}


def _wq(sd, name, scale=None):
    """bf16(fp32(w) * scale) in float64, as the backward pack rounds it."""
    w = sd[name + ".weight"].float()
    if scale is not None:
        w = w * torch.tensor(scale, dtype=torch.float32, device=w.device)
    return _bf(w).double()


def _block_w(sd, pre, s, nf, gc):
    """Forward-orientation weight of x_s -> [y | x4 .. x_{s+1}] of one dense block: the input gradient of x_s is its transpose."""
    lo, width = (nf + (s - 1) * gc, gc) if s else (0, nf)
    rows = [_wq(sd, f"{pre}.conv5", 0.2)] + [_wq(sd, f"{pre}.conv{j}") for j in range(4, s, -1)]
    return torch.cat([r[:, lo:lo + width] for r in rows], 0)


def _gate(act, neg):
    return torch.where(act > 0, torch.ones_like(act), torch.full_like(act, neg))


def _im2col(g, k):
    """(n, 1, H, W) -> (n, k*k, H, W): channel dy*k + dx = g at (y - dy + k//2, x - dx + k//2), zero outside (gcol_pack_kernel)."""
    p = k // 2
    hh, ww = g.shape[2:]
    gp = F.pad(g, (p, p, p, p))
    return torch.cat([gp[:, :, 2 * p - dy:2 * p - dy + hh, 2 * p - dx:2 * p - dx + ww] for dy in range(k) for dx in range(k)], 1)


def _drop_in(w):
    """w without the centre tap of one of its output channels, i.e. one input channel of the transposed conv."""
    w = w.clone()
    ky, kx = w.shape[2] // 2, w.shape[3] // 2
    w[int(w[:, :, ky, kx].abs().amax(1).argmax()), :, ky, kx] = 0
    return w


def _vjp(fn, shape, g):
    x = torch.zeros(shape, dtype=torch.float64, device=g.device, requires_grad=True)
    with torch.enable_grad():
        return torch.autograd.grad(fn(x), x, g)[0]


def _up_phase(x, wp, a, b, circular):
    """Phase (a, b) of nearest-x2 + 3x3 conv as the 2x2 conv over the low-resolution input."""
    h, wd = x.shape[2:]
    xp = F.pad(x, (1, 1, 1, 1), mode="circular" if circular else "constant")
    return F.conv2d(xp[:, :, a:a + h + 1, b:b + wd + 1], wp)


def _dgrad_lin(g, w, kind, shape, circular=False, drop=False, absolute=False):
    """Input gradient of the layer's linear map at g (absolute: sum |w||g|); with the cumulative phase partials for kind 'up'."""
    if absolute:
        g = g.abs()
    if kind == "up":
        total, partials = 0, []
        for (a, b), wp in w.items():
            wp = _drop_in(wp) if drop else wp
            wp = wp.abs() if absolute else wp
            total = total + _vjp(lambda x: _up_phase(x, wp, a, b, circular), shape, g[:, :, a::2, b::2])   # noqa: B023
            partials.append(total)
        return total, partials[:-1]
    w = _drop_in(w) if drop else w
    w = w.abs() if absolute else w
    pad = (w.shape[2] // 2, w.shape[3] // 2)
    return _vjp(lambda x: _conv(x, w, None, pad, circular), shape, g), []


def _wgrad_lin(x, g, shape, kind, circular):
    """sum over pixels of x (shifted by each tap) times g, float64: the weight gradient of the layer's forward."""
    co, ci, kh, kw = shape
    if kind == "up":
        x = F.interpolate(x, scale_factor=2, mode="nearest")
    if kind == "fold":                       # 9x1 conv over the x-im2col channels dx*ci + c
        if circular:
            x = F.pad(x, (0, 0, kh // 2, kh // 2), mode="circular")
        dw = conv2d_weight(x, (co, kw * ci, kh, 1), g, padding=(0 if circular else kh // 2, 0))
        return dw.reshape(co, kw, ci, kh).permute(0, 2, 3, 1)
    if circular:
        x = F.pad(x, (kw // 2, kw // 2, kh // 2, kh // 2), mode="circular")
        return conv2d_weight(x, shape, g)
    return conv2d_weight(x, shape, g, padding=(kh // 2, kw // 2))


class Checker:
    """The per-op checks of one backward; keeps the names checked and the worst ratio per op class (for calibration)."""

    def __init__(self, sd, controls):
        self.sd, self.controls = sd, controls
        self.dgrads, self.wgrads, self.worst = [], [], {}

    def _record(self, name, ratio, what):
        worst = float(ratio.max()) if ratio.numel() else 0.0
        if worst > self.worst.get(what, (0.0, ""))[0]:
            self.worst[what] = (worst, name)
        if not worst <= 1.0:
            i = int(torch.nan_to_num(ratio, nan=float("inf")).argmax())
            at = tuple(int(v) for v in torch.unravel_index(torch.tensor(i), ratio.shape))
            raise AssertionError(f"{name}: worst error / bound {worst:.3g} at {at}")

    def dgrad(self, name, got, g, w, kind="conv", gate=None, res=()):
        """got = gate * (transposed conv of g + residuals), NCHW float64; w in the forward orientation (cout = g's channels)."""
        n, c, hh, ww = got.shape
        shape = (n, c, hh, ww)
        a = _dgrad_lin(g, w, kind, shape, absolute=True)[0]
        v, partials = _dgrad_lin(g, w, kind, shape)
        gt = 1.0 if gate is None else gate
        ref = gt * (v + sum(res))
        tol = _ulp(ref) + REL * (gt * a + sum(r.abs() for r in res)) + sum(_ulp(p) for p in partials)
        tol = tol.clamp_min(1e-300)

        def ratio(circular=False, drop=False, ungated=False):
            r = ref
            if circular or drop or ungated:
                vv = _dgrad_lin(g, w, kind, shape, circular, drop)[0]
                r = (1.0 if ungated else gt) * (vv + sum(res))
            return (got - r).abs() / tol

        self._record(name, ratio(), "dgrad-phases" if kind == "up" else "dgrad")
        self.dgrads.append(name)
        if not self.controls:
            return
        k = 2 if kind == "up" else w.shape[2]
        if k > 1:
            r = ratio(circular=True)
            assert float(torch.cat([r[:, :, :1], r[:, :, -1:]], 2).max()) > 1.0, f"{name}: circular padding not detected on edge rows"
            assert float(torch.cat([r[..., :1], r[..., -1:]], 3).max()) > 1.0, f"{name}: circular padding not detected on edge columns"
        assert float(ratio(drop=True).max()) > 1.0, f"{name}: dropped tap not detected"
        if gate is not None:
            assert float(ratio(ungated=True).max()) > 1.0, f"{name}: gate replaced by 1 not detected"

    def wgrad(self, name, dw, db, terms, kind="conv", scale=1.0):
        """dw = scale sum_terms sum_pixels x g over the taps, db = scale sum g;  terms: (x, g[, g for db]) NCHW float64."""
        shape = tuple(dw.shape)

        def ref(circular=False, last=False, absolute=False):
            rw, rb = 0, 0
            for t in terms:
                x, g, gb = t if len(t) == 3 else (*t, t[1])
                if last:
                    x, g, gb = x[:-1], g[:-1], gb[:-1]
                if absolute:
                    x, g, gb = x.abs(), g.abs(), gb.abs()
                rw = rw + _wgrad_lin(x, g, shape, kind, circular)
                rb = rb + gb.sum((0, 2, 3))
            return scale * rw, scale * rb

        aw, ab = ref(absolute=True)
        tw, tb = (REL * aw).clamp_min(1e-300), (REL * ab).clamp_min(1e-300)

        def ratios(**kw):
            rw, rb = ref(**kw)
            return (dw - rw).abs() / tw, (db - rb).abs() / tb

        rw, rb = ratios()
        self._record(name + " dW", rw, "dW")
        self._record(name + " db", rb, "db")
        self.wgrads.append(name)
        if not self.controls:
            return
        if shape[2] > 1 or shape[3] > 1:
            assert float(ratios(circular=True)[0].max()) > 1.0, f"{name}: circular padding not detected in dW"
        if terms[0][0].shape[0] > 1:
            rw, rb = ratios(last=True)      # (db of a one-channel layer is one sum: one image's share can sit inside its bound)
            assert max(float(rw.max()), float(rb.max())) > 1.0, f"{name}: last image left out not detected in dW / db"


# (id, in_ch, nb, gc, n, h, w, options, controls, zero block in dL/dout)
CASES = [
    ("train-cfg3", 4, 11, 16, 16, 32, 32, {}, True, True),                  # bench.py --mode train
    ("train-gc32-w64", 4, 2, 32, 1, 64, 64, {}, True, False),               # per-layer weight gradients, 192-channel concat
    ("train-cfg4", 3, 2, 16, 1, 113, 113, {}, True, False),                 # ragged last windows, HR width 452
    ("train-tiny-dense", 1, 1, 16, 1, 9, 7, {31: 0}, False, False),         # raster smaller than one window, dense kernel forced
    ("train-halo-w64", 4, 1, 16, 3, 37, 64, {37: 0}, False, False),         # halo-column tiling on a 64-wide map, ragged height
    ("train-layer-dgrads", 4, 2, 16, 2, 24, 40, {27: 0, 25: 0}, True, False),   # narrow input gradients as per-layer convs,
                                                                                # deterministic weight gradients (reduce kernel)
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_generator_backward_layers_match_float64(case):
    from climsr_b200._lib import check, current_stream_ptr, lib
    from oracle import synth
    cid, in_ch, nb, gc, n, h, w, opts, controls, zero_block = case
    nf = 64
    with _options(opts):
        net, sd, x, _elev, _mask, _sr = _run(in_ch, nb, gc, n, h, w, True, seed=61)
        buf = PlanBuffers(net, n, h, w, True)
        gen = torch.Generator().manual_seed(67)
        go = torch.rand((n, 1, 4 * h, 4 * w), generator=gen) * 2 - 1
        if zero_block:                           # land-masked pixels give exact zeros; this block touches the top and left edges
            go[0, :, :2 * h, :4 * w // 3] = 0
        go = go.cuda().contiguous()
        packed_bwd = net.packed_weights_bwd(force=True)
        plan = buf.plan
        nfloat = lib.csr_plan_grad_floats(plan)
        offs = net._grad_offsets(plan)
        specs = synth.conv_specs(in_ch, 1, nf, nb, gc)
        names = [s[0] for s in specs]
        base_tail = 1 + 15 * nb

        def grads(li):
            _, co, ci, kh, kw = specs[li]
            o, ob = offs[2 * li], offs[2 * li + 1]
            return flat[o:o + co * ci * kh * kw].view(co, ci, kh, kw).double(), flat[ob:ob + co].double()

        ck = Checker(sd, controls)
        f = lambda kind, i=0: _nchw(buf(kind, i))     # noqa: E731  forward activations (the backward does not write them)
        hrA, hrB, hrD, hrE, hrC, m1, t0 = f(2), f(3), f(4), f(5)[:, :32], f(8)[:, :27], f(1), f(7)
        gbf = _bf(go.double())

        # ---- the stops: (lowest layer completed, check(prev, cur)) ------------------------------------------------------------
        def tail0(p, s):
            assert torch.equal(s["gO"][:, :25], _im2col(gbf, 5)), "gO differs from the 5x5 im2col of bf16(dL/dout)"
            assert bool((s["gO"][:, 25:] == 0).all()), "gO: padding channels 25..31 not zero"
            ck.wgrad("srcnn.conv3", *grads(base_tail + 7), [(hrE, gbf, go.double())])

        def tail1(p, s):
            ck.dgrad("srcnn.conv3.dgrad_cols", s["gP"][:, :32], gbf, _wq(sd, "srcnn.conv3"), gate=_gate(hrE, 0.0))
            ck.wgrad("srcnn.conv2", *grads(base_tail + 6), [(hrD, s["gP"][:, :32])])

        def tail2(p, s):
            ck.dgrad("srcnn.conv2.dgrad", s["gQ"], p["gP"][:, :32], _wq(sd, "srcnn.conv2"), gate=_gate(hrD, 0.0))
            ck.wgrad("srcnn.conv1", *grads(base_tail + 5), [(hrC, s["gQ"])], kind="fold")

        def tail3(p, s):
            ck.dgrad("srcnn.conv1.dgrad", s["gT"][:, :3], p["gQ"], _wq(sd, "srcnn.conv1"))
            assert torch.equal(s["gcolB"][:, :9], _im2col(s["gT"][:, :1], 3)), "gcolB differs from the 3x3 im2col of gT channel 0"
            assert bool((s["gcolB"][:, 9:] == 0).all()), "gcolB: padding channels 9..15 not zero"
            ck.wgrad("conv_last", *grads(base_tail + 4), [(hrB, s["gT"][:, :1])])

        def tail4(p, s):
            ck.dgrad("conv_last.dgrad_cols", s["gP"], p["gT"][:, :1], _wq(sd, "conv_last"), gate=_gate(hrB, 0.2))
            ck.wgrad("HRconv", *grads(base_tail + 3), [(hrA, s["gP"])])

        def tail5(p, s):
            ck.dgrad("HRconv.dgrad", s["gQ"], p["gP"], _wq(sd, "HRconv"), gate=_gate(hrA, 0.2))
            ck.wgrad("upconv2", *grads(base_tail + 2), [(m1, s["gQ"])], kind="up")

        def tail6(p, s):
            ck.dgrad("upconv2.dgrad", s["gm1"], p["gQ"], _phase_weights(sd["upconv2.weight"]), kind="up", gate=_gate(m1, 0.2))
            ck.wgrad("upconv1", *grads(base_tail + 1), [(t0, s["gm1"])], kind="up")

        def tail7(p, s):
            ck.dgrad("upconv1.dgrad", s["gt0"], p["gm1"], _phase_weights(sd["upconv1.weight"]), kind="up")
            ck.wgrad("trunk_conv", *grads(base_tail), [(f(0, 3 * nb)[:, :nf], s["gt0"])])

        stops = [(base_tail + 7 - t, fn) for t, fn in enumerate((tail0, tail1, tail2, tail3, tail4, tail5, tail6, tail7))]

        # dense blocks in the order bwd_build runs them, with its buffer rotation
        blocks, Pb = [], 0
        for i in range(nb - 1, -1, -1):
            Qb, Rb = (Pb + 1) % 3, (Pb + 2) % 3
            for r, gb, xo in ((2, Qb, Rb), (1, Rb, Qb), (0, Qb, Rb)):
                blocks.append(dict(i=i, r=r, Gb=gb, Xo=xo, Pb=Pb, Qb=Qb))
            Pb = Rb
        cw = nf + 4 * gc

        def wide(p, s, blk):
            """The block's input gradient: conv_T(Gb) + g_y (+ G for an RDB1), into the next Gb[:64]."""
            pre = f"RRDB_trunk.{blk['i']}.RDB{blk['r'] + 1}"
            gb = p["cat"][blk["Gb"]]
            res = (gb[:, :nf],) + ((p["cat"][blk["Pb"]][:, :nf],) if blk["r"] == 0 else ())
            ck.dgrad(f"{pre}.conv5.dgrad_x0", s["cat"][blk["Xo"]][:, :nf], gb[:, :cw], _block_w(sd, pre, 0, nf, gc), res=res)

        def block_stop(b):
            blk = blocks[b]

            def fn(p, s):
                if b == 0:
                    ck.dgrad("trunk_conv.dgrad", s["cat"][0][:, :nf], p["gt0"], _wq(sd, "trunk_conv"))
                else:
                    wide(p, s, blocks[b - 1])
                if blk["r"] == 2:
                    want = _bf(s["cat"][blk["Pb"]][:, :nf].float() * torch.tensor(0.2, dtype=torch.float32, device="cuda")).double()
                    assert torch.equal(s["cat"][blk["Qb"]][:, :nf], want), "kScale: RDB3's g_y differs from bf16(0.2f G)"
                i, r = blk["i"], blk["r"]
                pre = f"RRDB_trunk.{i}.RDB{r + 1}"
                gb = s["cat"][blk["Gb"]]
                xcat = f(0, 3 * i + r)
                for sidx in range(4, 0, -1):
                    lo = nf + (4 - sidx) * gc
                    ck.dgrad(f"{pre}.conv5.dgrad_x{sidx}", gb[:, lo:lo + gc], gb[:, :lo], _block_w(sd, pre, sidx, nf, gc),
                             gate=_gate(xcat[:, nf + (sidx - 1) * gc:nf + sidx * gc], 0.2))
                for k in range(1, 5):
                    lo = nf + (4 - k) * gc
                    ck.wgrad(f"{pre}.conv{k}", *grads(1 + (3 * i + r) * 5 + k - 1), [(xcat[:, :nf + (k - 1) * gc], gb[:, lo:lo + gc])])
                ck.wgrad(f"{pre}.conv5", *grads(1 + (3 * i + r) * 5 + 4), [(xcat[:, :cw], gb[:, :nf])], scale=0.2)
            return 1 + (3 * blk["i"] + blk["r"]) * 5, fn

        stops += [block_stop(b) for b in range(len(blocks))]

        def last(p, s):
            wide(p, s, blocks[-1])
            xin = _bf(x.cuda().double())
            ck.wgrad("conv_first", *grads(0), [(xin, s["cat"][Pb][:, :nf]), (xin, s["gt0"])])

        stops.append((0, last))

        # ---- run the backward stop by stop -----------------------------------------------------------------------------------
        nseg = lib.csr_plan_backward_segments(plan, nfloat)
        check(min(nseg, 0), "csr_plan_backward_segments")
        assert nseg == len(stops) == 8 + 3 * nb + 1, f"{nseg} backward segments, expected one per layer-completion point ({len(stops)})"
        flat = torch.full((nfloat,), float("nan"), device="cuda")
        lo, hi = C.c_size_t(), C.c_size_t()
        prev, prev_lo = None, nfloat
        for k, (layer, fn) in enumerate(stops):
            check(lib.csr_plan_backward_flat_seg(plan, packed_bwd.data_ptr(), go.data_ptr(), flat.data_ptr(), k, C.byref(lo), C.byref(hi),
                                                 current_stream_ptr()), "csr_plan_backward_flat_seg")
            torch.cuda.synchronize()
            assert (lo.value, hi.value) == (offs[2 * layer], prev_lo), f"segment {k}: gradient floats [{lo.value}, {hi.value}), " \
                f"expected [{offs[2 * layer]}, {prev_lo}) ({names[layer]} and the layers after it)"
            prev_lo = lo.value
            cur = {name: _nchw(buf(kind)) for name, kind in GRAD_KINDS.items()}
            cur["cat"] = [_nchw(buf(17, j)) for j in range(3)]
            fn(prev, cur)
            prev = cur
        assert not torch.isnan(flat).any(), "the segments left part of the flat gradient buffer unwritten"

        if opts.get(25) == 0:
            # weight gradients through per-CTA slices and the reduce kernel: the segmented backward is the whole backward bit for
            # bit, up to the bias reductions, which add with atomics in a run-dependent order
            whole = torch.full_like(flat, float("nan"))
            check(lib.csr_plan_backward_flat(plan, packed_bwd.data_ptr(), go.data_ptr(), whole.data_ptr(), current_stream_ptr()),
                  "csr_plan_backward_flat")
            torch.cuda.synchronize()
            _assert_same_flat(flat, whole, _flat_layout(net, plan))

    bwd_names = ["srcnn.conv3.dgrad_cols", "srcnn.conv2.dgrad", "srcnn.conv1.dgrad", "conv_last.dgrad_cols", "HRconv.dgrad",
                 "upconv2.dgrad", "upconv1.dgrad", "trunk_conv.dgrad"]
    bwd_names += [f"RRDB_trunk.{i}.RDB{r}.conv5.dgrad_x{s}" for i in range(nb) for r in (1, 2, 3) for s in range(5)]
    assert sorted(ck.dgrads) == sorted(bwd_names)            # every input-gradient layer (bwd_layer_table) exactly once
    assert sorted(ck.wgrads) == sorted(names)                # every layer's dW / db exactly once
    print(f"{cid}: {nseg} stops, {len(ck.dgrads)} input gradients, {len(ck.wgrads)} weight gradients, worst error / bound",
          {k: (round(v[0], 3), v[1]) for k, v in ck.worst.items()})


def test_gradient_buffers_exist_in_training_plans_only():
    from climsr_b200._lib import CSR_ERR_BAD_ARG, CSR_OK, lib
    n, h, w = 1, 9, 7
    off, dims = C.c_size_t(), (C.c_int32 * 4)()
    for train in (False, True):
        net = _run(1, 1, 16, n, h, w, train, seed=61)[0]
        plan = PlanBuffers(net, n, h, w, train).plan
        for kind in range(10, 18):
            rc = lib.csr_plan_buffer(plan, kind, 0, C.byref(off), C.byref(dims))
            assert rc == (CSR_OK if train else CSR_ERR_BAD_ARG), f"kind {kind}, train {train}: rc {rc}"
            if train:
                s = 4 if kind <= 14 else 2 if kind == 15 else 1
                assert tuple(dims)[:3] == (n, s * h, s * w)
        for kind, index in ((17, -1), (17, 3), (18, 0)):
            assert lib.csr_plan_buffer(plan, kind, index, C.byref(off), C.byref(dims)) == CSR_ERR_BAD_ARG, (train, kind, index)
