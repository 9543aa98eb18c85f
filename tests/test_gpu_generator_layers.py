"""Every launch of the generator forward, read back from the plan's own buffers (csr_plan_buffer) and held element by element to a
float64 recomputation of the same layer from the operands that launch read.

Reference of a layer: the bf16 operands as stored in the plan, bf16(w) (the pack kernel rounds the fp32 weights once, RNE) and the
fp32 bias unrounded, in float64, with the layer's epilogue (LeakyReLU(0.2) / ReLU; RDB conv5 (acc + b) 0.2 + r1; RDB3 conv5
((acc + b) 0.2 + r1) 0.2 + r2; trunk_conv acc + b + fea0).  upconv1 / upconv2 are recomputed in the sub-pixel form the kernel
executes: phase (a, b) is a 2x2 conv over the low-resolution input whose taps are bf16(fp32 sums of the 3x3 taps mapped to them),
summed in the pack kernel's order (elementwise.cu phase_taps).  srcnn.conv1 is the 9x1 conv over the x-im2col input (kind 8).

Bound, per element:  |got - ref| <= ulp_bf16(ref) + 2^-12 A  (fp32 outputs: no ulp term), where A is the epilogue applied to
absolute values: scale (sum |w||x| + |b|) + scale2 |r1| + |r2|.  The ulp term is the bf16 store (half an ulp, one when the fp32
accumulator straddles a rounding boundary); 2^-12 A is far above fp32 accumulation noise and far below one missing product.
Measured on a B200 (1000 W power limit), worst error / bound over all cases: 0.483 at bf16 outputs (RDB3 conv5: the store rounds
the fp32 accumulator, half an ulp), below 5e-4 at fp32 outputs (conv_last in training, srcnn.conv3).

Inference plans keep neither HRconv's output nor srcnn.conv1's (their epilogues run the next layer as a second MMA over the
staged bf16 tile), so two composites are checked there: hrA -> hrC (HRconv, conv_last's nine tap planes, tap_pack) and hrC ->
hrE (srcnn.conv1, srcnn.conv2).  Their reference rounds the inner activation to bf16 as the staged tile does; where the kernel's
fp32 accumulator and the float64 value straddle a rounding boundary the two inner values are one bf16 ulp apart, so the bound adds
k * sum |w_outer| ulp(inner) with k = 1/4 (a small share of the inner values flips, with random signs).  Measured on the same
B200: worst 0.833 (srcnn.conv1 + srcnn.conv2 at the cfg2 batch); k = 1/8 was exceeded (1.31).

Sensitivity controls (reference side only): at W = 32, 64 and a ragged width, the same reference with circular instead of zero
padding must break the bound on the edge rows and columns, and one with one input channel of one tap dropped must break it too.
"""
import ctypes as C
from contextlib import contextmanager

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

REL = 2.0 ** -12
K_INNER = 1.0 / 4
OPTION_DEFAULTS = {25: 1, 27: 1, 31: 2, 33: 3, 36: 1, 37: 1}


@contextmanager
def _options(opts):
    """Plan-creation options (csr_set_option), back to the library defaults afterwards."""
    from climsr_b200._lib import lib
    try:
        for k, v in opts.items():
            lib.csr_set_option(k, v)
        yield
    finally:
        for k, v in OPTION_DEFAULTS.items():
            lib.csr_set_option(k, v)


def _bf(t):
    return t.to(torch.bfloat16).to(t.dtype)


def _ulp(v):
    """Spacing of bf16 values at |v| (0 at v = 0)."""
    _, e = torch.frexp(v)
    return torch.where(v == 0, torch.zeros_like(v), torch.pow(2.0, (e - 8).to(v.dtype)))


def _nchw(t):
    return t.permute(0, 3, 1, 2).double()


# ---------------------------------------------------------------------------------------------------------------- references
def _conv(x, w, b, pad, circular):
    if circular:
        return F.conv2d(F.pad(x, (pad[1], pad[1], pad[0], pad[0]), mode="circular"), w, b)
    return F.conv2d(x, w, b, padding=pad)


def _phase_weights(w):
    """The four 2x2 sub-pixel weights of nearest-x2 + 3x3 conv: fp32 sums in the pack kernel's (yy, xx) order, then bf16."""
    taps = {0: ((0, 0), (1, 2)), 1: ((0, 1), (2, 2))}           # a -> (range of 3x3 rows feeding tap row 0, tap row 1)
    out = {}
    for a in (0, 1):
        for b in (0, 1):
            wp = torch.zeros(w.shape[:2] + (2, 2), dtype=torch.float32, device=w.device)
            for ry in (0, 1):
                for rx in (0, 1):
                    y0, y1 = taps[a][ry]
                    x0, x1 = taps[b][rx]
                    v = torch.zeros(w.shape[:2], dtype=torch.float32, device=w.device)
                    for yy in range(y0, y1 + 1):
                        for xx in range(x0, x1 + 1):
                            v = v + w[:, :, yy, xx]
                    wp[:, :, ry, rx] = v
            out[(a, b)] = _bf(wp).double()
    return out


def _drop_tap(w):
    """w without one input channel of its centre tap (the channel with the largest weight there)."""
    w = w.clone()
    ky, kx = w.shape[2] // 2, w.shape[3] // 2
    w[:, int(w[:, :, ky, kx].abs().amax(0).argmax()), ky, kx] = 0
    return w


def _linear(x, w, b, kind, circular=False, drop=False, absolute=False):
    """acc + b of one launch in float64 (absolute: sum |w||x| + |b|)."""
    w = w.to(x.device)
    b = b.to(x.device).double()
    if absolute:
        x = x.abs()
        b = b.abs()
    if kind == "up":
        ws = _phase_weights(w)
        n, _, h, wd = x.shape
        out = torch.empty((n, w.shape[0], 2 * h, 2 * wd), dtype=torch.float64, device=x.device)
        xp = F.pad(x, (1, 1, 1, 1), mode="circular" if circular else "constant")
        for (a, bb), wp in ws.items():
            if drop:
                wp = _drop_tap(wp)
            out[:, :, a::2, bb::2] = F.conv2d(xp[:, :, a:a + h + 1, bb:bb + wd + 1], wp.abs() if absolute else wp, b)
        return out
    if kind == "fold":                       # srcnn.conv1: 9x1 over the im2col channels dx*3 + c
        co, ci, kh, kw = w.shape
        wq = _bf(w).double().permute(0, 3, 1, 2).reshape(co, kw * ci, kh, 1)
        pad = (kh // 2, 0)
    else:
        wq = _bf(w).double()
        pad = (w.shape[2] // 2, w.shape[3] // 2)
    if drop:
        wq = _drop_tap(wq)
    return _conv(x, wq.abs() if absolute else wq, b, pad, circular)


def _epilogue(v, act, res, absolute=False):
    if act == "lrelu" and not absolute:
        v = F.leaky_relu(v, 0.2)
    elif act == "relu" and not absolute:
        v = F.relu(v)
    for s, r in res:
        v = v * s + (r.abs() if absolute else r)
    return v


def _ratio(got, ref, a, fp32=False, extra=None):
    tol = REL * a
    if not fp32:
        tol = tol + _ulp(ref)
    if extra is not None:
        tol = tol + extra
    return (got - ref).abs() / tol.clamp_min(1e-300)


class Checker:
    """Runs the per-layer checks of one plan and keeps the names checked and the worst ratio (for calibration)."""

    def __init__(self, sd, dev, controls):
        self.sd, self.dev, self.controls = sd, dev, controls
        self.names, self.worst = [], {}

    def _record(self, names, ratio, what):
        worst = float(ratio.max())
        if worst > self.worst.get(what, (0.0, ""))[0]:
            self.worst[what] = (worst, "+".join(names))
        if not worst <= 1.0:
            i = int(torch.nan_to_num(ratio, nan=float("inf")).argmax())
            n_, c_, y_, x_ = (int(v) for v in torch.unravel_index(torch.tensor(i), ratio.shape))
            raise AssertionError(f"{'+'.join(names)}: worst error / bound {worst:.3g} at (n, y, x, c) = ({n_}, {y_}, {x_}, {c_})")
        self.names += names

    def _controls(self, name, ratio_fn, rows, cols):
        """The circular-padding and dropped-tap references must break the bound (at the edges for the former)."""
        if not self.controls:
            return
        if rows or cols:
            r = ratio_fn(circular=True)
            if rows:
                assert float(torch.cat([r[:, :, :1], r[:, :, -1:]], 2).max()) > 1.0, f"{name}: circular padding not detected on edge rows"
            if cols:
                assert float(torch.cat([r[..., :1], r[..., -1:]], 3).max()) > 1.0, f"{name}: circular padding not detected on edge columns"
        assert float(ratio_fn(drop=True).max()) > 1.0, f"{name}: dropped tap not detected"

    def layer(self, name, x, got, kind="conv", act=None, res=(), fp32=False):
        """One launch: x, got NCHW float64 (operands / results as stored), res = ((scale, residual), ...)."""
        w, b = self.sd[name + ".weight"], self.sd[name + ".bias"]
        x, got = x.to(self.dev), got.to(self.dev)
        res = tuple((s, r.to(self.dev)) for s, r in res)
        a = _epilogue(_linear(x, w, b, kind, absolute=True), act, res, absolute=True)

        def ratio(circular=False, drop=False):
            return _ratio(got, _epilogue(_linear(x, w, b, kind, circular, drop), act, res), a, fp32)

        self._record([name], ratio(), "fp32" if fp32 else "bf16")
        kh, kw = w.shape[2:]
        self._controls(name, ratio, rows=kh > 1, cols=kw > 1 and kind != "fold")

    def composite(self, inner, outer, x, inner_kind, inner_act, outer_act, finish, got):
        """inner -> bf16 -> outer, intermediate not stored.  finish(v) maps the outer result onto the stored layout of `got`."""
        wi, bi = self.sd[inner + ".weight"], self.sd[inner + ".bias"]
        wo, bo = self.sd[outer + ".weight"], self.sd[outer + ".bias"]
        x, got = x.to(self.dev), got.to(self.dev)
        pad = (wo.shape[2] // 2, wo.shape[3] // 2)
        wabs = _bf(wo.to(self.dev)).double().abs()

        def ratio(circular=False, drop=False):
            mid = _bf(_epilogue(_linear(x, wi, bi, inner_kind, circular), inner_act, ()))
            ref = _epilogue(_linear(mid, wo, bo, "conv", drop=drop), outer_act, ())
            a = _linear(mid, wo, bo, "conv", absolute=True)
            extra = K_INNER * F.conv2d(_ulp(mid), wabs, None, padding=pad)
            return _ratio(got, finish(ref), finish(a), extra=finish(extra))

        self._record([inner, outer], ratio(), "composite")
        self._controls(inner + "+" + outer, ratio, rows=True, cols=inner_kind != "fold")


def _im2col_x(t):
    """(n, c, H, W) -> (n, 9c, H, W): channel dx*c + ci = t[:, ci] at x + dx - 4, zero outside the image."""
    wd = t.shape[3]
    p = F.pad(t, (4, 4))
    return torch.cat([p[..., dx:dx + wd] for dx in range(9)], 1)


# ---------------------------------------------------------------------------------------------------------------- plan buffers
class PlanBuffers:
    def __init__(self, net, n, h, w, train):
        from climsr_b200._lib import check, lib
        self.check, self.lib = check, lib
        (self.plan, self.ws), = [v for k, v in net._plans.items() if k[:3] == (n, h, w) and k[4] == train]
        self.base = (self.ws.data_ptr() + 1023) // 1024 * 1024 - self.ws.data_ptr()

    def __call__(self, kind, index=0):
        """NHWC view (bf16; kind 9: fp32) of buffer `kind` as csr_plan_buffer documents it."""
        off, dims = C.c_size_t(), (C.c_int32 * 4)()
        self.check(self.lib.csr_plan_buffer(self.plan, kind, index, C.byref(off), C.byref(dims)), "csr_plan_buffer")
        shape = tuple(int(v) for v in dims)
        dt, es = (torch.float32, 4) if kind == 9 else (torch.bfloat16, 2)
        nbytes = shape[0] * shape[1] * shape[2] * shape[3] * es
        lo = self.base + off.value
        return self.ws[lo:lo + nbytes].view(dt).view(shape)


def _run(in_ch, nb, gc, n, h, w, train, seed):
    from climsr_b200.models import ESRGANGenerator
    from oracle import synth
    sd = synth.make_state_dict(in_ch, 1, 64, nb, gc, seed=seed, gain=1.3)
    x, elev, mask = synth.make_inputs(n, in_ch, h, w, seed=seed + 1)
    net = ESRGANGenerator(in_ch, 1, 64, nb, gc)
    net.load_state_dict(sd)
    net = net.cuda().train(train)
    with torch.set_grad_enabled(train):
        sr = net(x.cuda(), elev.cuda(), mask.cuda())
    torch.cuda.synchronize()
    assert torch.isfinite(sr).all()
    return net, {k: v.cuda() for k, v in sd.items()}, x, elev, mask, sr.detach()


def _check_trunk(ck, buf, nb, gc, train, first_rrdb, x_in):
    """conv_first and the RRDB layers whose operands survive the forward, then trunk_conv."""
    fea0 = _nchw(buf(6))
    ck.layer("conv_first", _bf(x_in.cuda().double()), fea0)
    if train:
        assert torch.equal(buf(0, 0)[..., :64], buf(6)), "conv_first: concat 0 and fea0 differ"
    cat = lambda j: _nchw(buf(0, j if train else j % 3))    # noqa: E731
    for i in range(first_rrdb, nb):
        rrdb_in = fea0 if (not train and nb == 1) else cat(3 * i)[:, :64]
        for r in range(3):
            j = 3 * i + r
            src = cat(j)
            if not train and r == 0:
                if nb > 1:
                    continue                    # x of the last RRDB's RDB1 is overwritten by its output
                src = torch.cat([fea0, src[:, 64:]], 1)
            pre = f"RRDB_trunk.{i}.RDB{r + 1}"
            for k in range(1, 5):
                ck.layer(f"{pre}.conv{k}", src[:, :64 + (k - 1) * gc], src[:, 64 + (k - 1) * gc:64 + k * gc], act="lrelu")
            if not train and r == 2 and nb > 1:
                continue                        # its second residual, the RRDB input, is gone
            dst = cat(j + 1) if (train or r < 2) else cat(3 * i)
            res = ((0.2, src[:, :64]),) + (((0.2, rrdb_in),) if r == 2 else ())
            ck.layer(f"{pre}.conv5", src[:, :64 + 4 * gc], dst[:, :64], res=res)
    trunk_in = cat(3 * nb)[:, :64] if train else cat(0)[:, :64]
    ck.layer("trunk_conv", trunk_in, _nchw(buf(7)), res=((1.0, fea0),))


def _check_tail(ck, buf, train, elev, mask, sr, sel):
    """upconv1 .. srcnn.conv3 on the images `sel`."""
    pick = lambda t: t[sel]                 # noqa: E731
    ck.layer("upconv1", pick(_nchw(buf(7))), pick(_nchw(buf(1))), kind="up", act="lrelu")
    hra = pick(_nchw(buf(2)))
    ck.layer("upconv2", pick(_nchw(buf(1))), hra, kind="up", act="lrelu")
    hrc = pick(buf(8)).permute(0, 3, 1, 2)
    pitch = hrc.shape[1]
    e, m = (_bf(pick(t).cuda()).double() for t in (elev, mask))
    # channels 27..31 pad srcnn.conv1's 27 input channels to 32; training plans leave 32..63 of their 64-channel pitch unwritten
    assert bool((hrc[:, 27:min(32, pitch)] == 0).all()), "SRCNN input: padding channels 27..31 not zero"
    hrc = hrc.double()
    if train:
        hrb = _nchw(pick(buf(3)))
        ck.layer("HRconv", hra, hrb, act="lrelu")
        t = pick(buf(9)).permute(0, 3, 1, 2).double()
        ck.layer("conv_last", hrb, t, fp32=True)
        want = _im2col_x(torch.cat([_bf(t), e, m], 1))
        assert torch.equal(hrc[:, :27], want), "SRCNN input im2col differs from bf16 of (conv_last, elev, mask)"
        hrd = _nchw(pick(buf(4)))
        ck.layer("srcnn.conv1", hrc[:, :27], hrd, kind="fold", act="relu")
        hre = _nchw(pick(buf(5)))[:, :32]
        ck.layer("srcnn.conv2", hrd, hre, act="relu")
    else:
        em = _im2col_x(torch.cat([torch.zeros_like(e), e, m], 1))
        assert torch.equal(hrc[:, :27].reshape(-1, 9, 3, *hrc.shape[2:])[:, :, 1:],
                           em.reshape(-1, 9, 3, *em.shape[2:])[:, :, 1:]), "SRCNN input: elev / mask channels differ"
        ck.composite("HRconv", "conv_last", hra, "conv", "lrelu", None, _im2col_x, hrc[:, 0:27:3])
        hre = _nchw(pick(buf(5)))[:, :32]
        ck.composite("srcnn.conv1", "srcnn.conv2", hrc[:, :27], "fold", "relu", "relu", lambda v: v, hre)
    ck.layer("srcnn.conv3", hre, pick(sr).double(), fp32=True)


# (id, train, in_ch, nb, gc, n, h, w, options, controls)
CASES = [
    ("train-cfg3", True, 4, 11, 16, 16, 32, 32, {}, True),              # bench.py --mode train: whole 32-pixel rows, ~175 layers
    ("train-gc32-w64", True, 4, 2, 32, 1, 64, 64, {}, True),            # per-layer convs, 192-channel concat, whole 64-pixel rows
    ("train-cfg4", True, 3, 2, 16, 1, 113, 113, {}, True),              # ragged last windows, HR width 452
    ("train-tiny-dense", True, 1, 1, 16, 1, 9, 7, {31: 0}, False),      # raster smaller than one window, dense kernel forced
    ("train-halo-w64", True, 4, 1, 16, 3, 37, 64, {37: 0}, False),      # halo-column tiling on a 64-wide map, ragged height
    ("infer-cfg2-nb1", False, 4, 1, 16, 64, 64, 64, {}, True),          # every trunk launch incl. the in-place RDB3 conv5
    ("infer-cfg2-nb11", False, 4, 11, 16, 64, 64, 64, {}, False),       # Hydra depth: what the rotating buffers still hold
    ("infer-cfg4", False, 3, 1, 16, 1, 113, 113, {}, False),            # tap_pack with two 256-pixel row segments
    ("infer-many-windows", False, 4, 1, 16, 150, 16, 16, {31: 0}, False),   # more windows than SMs
    ("infer-low-m-tile", False, 4, 1, 16, 2, 5, 33, {31: 0}, False),    # second M tile mostly below the image
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_generator_layers_match_float64(case):
    from oracle import synth
    cid, train, in_ch, nb, gc, n, h, w, opts, controls = case
    with _options(opts):
        net, sd, x, elev, mask, sr = _run(in_ch, nb, gc, n, h, w, train, seed=61)
        buf = PlanBuffers(net, n, h, w, train)
        ck = Checker(sd, "cuda", controls)
        _check_trunk(ck, buf, nb, gc, train, first_rrdb=0 if (train or nb == 1) else nb - 1, x_in=x)
        sel = [0, n // 2, n - 1] if n > 16 else list(range(n))    # the HR tail of the large inference batches: three images
        _check_tail(ck, buf, train, elev, mask, sr, sel)
    names = [s[0] for s in synth.conv_specs(in_ch, 1, 64, nb, gc)]
    if train or nb == 1:
        from climsr_b200._lib import NetDesc, lib
        assert sorted(ck.names) == sorted(names)                    # every layer has its own check ...
        assert len(ck.names) == lib.csr_num_layers(C.byref(NetDesc(in_ch, 1, 64, nb, gc, 4)))   # ... and only one
    else:
        last = [f"RRDB_trunk.{nb - 1}.RDB2.conv{k}" for k in range(1, 6)] + [f"RRDB_trunk.{nb - 1}.RDB3.conv{k}" for k in range(1, 5)]
        assert sorted(ck.names) == sorted(["conv_first"] + last + names[-8:])     # names[-8:]: trunk_conv .. srcnn.conv3
    print(f"{cid}: {len(ck.names)} layers, worst error / bound", {k: (round(v[0], 3), v[1]) for k, v in ck.worst.items()})
