"""Drop-in ``RCAN`` generator (the reference's default ``generator_type``, climsr/core/config.py:64) on the sm_100a kernels,
inference and training (SURVEY.md section 8f row 4).

Mirrors climsr/models/rcan.py:137-217: same constructor signature (``conv`` is accepted and must be the default), same
sub-module / parameter names (``head``, ``body.{g}.body.{b}.body.{0,2}`` + ``.body.3.conv_du.{0,2}``, ``tail.0.{0,2}``,
``tail.1``, ``srcnn.conv{1,2,3}``) and creation order - the parameter containers are plain nn.Conv2d - so
``load_state_dict`` (the reference's tolerant override included) and ``torch.manual_seed`` initialisation behave as before;
same ``forward(x, elev, mask) -> (N, 1, 4h, 4w)``.

Every 3x3 convolution runs on the tcgen05 conv kernel (csr_conv2d_nhwc) with bias / ReLU / the ResidualGroup and body
skip-adds fused in the epilogue; CALayer (global average pool -> 1x1 -> ReLU -> 1x1 -> sigmoid -> scale) together with the
RCAB skip is csr_channel_attention, PixelShuffle(2) is csr_pixel_shuffle2, the SRCNN tail runs on the same conv kernel.
Packed weights are cached per weight version.

Training: in ``train()`` mode with gradients enabled the forward runs the same launch sequence through ``_RCANFunction``,
which keeps the activations the backward needs on its autograd node (freed with the graph).  ``loss.backward()`` runs the
input-gradient convs on the same conv kernel (transposed packs, ReLU' as the epilogue gate, the skip gradients as epilogue
residuals), csr_channel_attention_backward for CALayer, csr_pixel_unshuffle2 for PixelShuffle, and csr_conv2d_wgrad for every
conv, and hands back ordinary fp32 ``.grad`` tensors (views of one zeroed buffer in ``parameters()`` order).  Gradients
w.r.t. x, elev and mask are not produced.  In ``eval()`` mode a forward under ``torch.enable_grad()`` with parameters that
require gradients raises, as it always has.  There is no CPU fallback.
"""
from __future__ import annotations

import logging
import math
from typing import Optional

import torch
import torch.nn as nn
from torch import Tensor

from .. import ops
from .._lib import CsrError, check, current_stream_ptr, lib
from ._common import DerivedState, _SRCNNParams, check_generator_inputs, f32, flat_grad_views


def default_conv(in_channels: int, out_channels: int, kernel_size: int, bias: bool = True) -> nn.Module:
    return nn.Conv2d(in_channels, out_channels, kernel_size, padding=kernel_size // 2, bias=bias)


class _CALayerParams(nn.Module):
    def __init__(self, channel: int, reduction: int = 16):
        super().__init__()
        self.avg_pool = nn.AdaptiveAvgPool2d(1)
        self.conv_du = nn.Sequential(nn.Conv2d(channel, channel // reduction, 1, padding=0, bias=True), nn.ReLU(inplace=True),
                                     nn.Conv2d(channel // reduction, channel, 1, padding=0, bias=True), nn.Sigmoid())


class _RCABParams(nn.Module):
    def __init__(self, n_feat: int, kernel_size: int, reduction: int):
        super().__init__()
        self.body = nn.Sequential(default_conv(n_feat, n_feat, kernel_size), nn.ReLU(True), default_conv(n_feat, n_feat, kernel_size),
                                  _CALayerParams(n_feat, reduction))
        self.res_scale = 1


class _ResidualGroupParams(nn.Module):
    def __init__(self, n_feat: int, kernel_size: int, reduction: int, n_resblocks: int):
        super().__init__()
        body = [_RCABParams(n_feat, kernel_size, reduction) for _ in range(n_resblocks)]
        body.append(default_conv(n_feat, n_feat, kernel_size))
        self.body = nn.Sequential(*body)


class RCAN(DerivedState, nn.Module):
    def __init__(self, n_resgroups: int = 10, n_resblocks: int = 20, n_feats: int = 64, reduction: int = 16, scaling_factor: int = 4,
                 in_channels: int = 3, out_channels: int = 1, conv=default_conv, **kwargs):
        super().__init__()
        if conv is not default_conv and conv is not None:
            raise ValueError("climsr_b200 RCAN supports the reference's default_conv only")
        if n_feats != 64 or scaling_factor != 4 or out_channels != 1 or not (1 <= in_channels <= 16) or n_feats % reduction:
            raise ValueError("climsr_b200 RCAN supports n_feats=64, scaling_factor=4, out_channels=1, 1<=in_channels<=16")
        self.n_resgroups, self.n_resblocks, self.n_feats = n_resgroups, n_resblocks, n_feats
        self.kernel_size, self.reduction, self.scaling_factor = 3, reduction, scaling_factor
        self.in_channels = in_channels
        # creation order of rcan.py:164-186 (body, then head ... the reference builds the lists first, then the Sequentials in the
        # order head, body, tail, srcnn; parameters are created when the conv objects are): head conv, groups, body conv, tail
        head = [default_conv(in_channels, n_feats, 3)]
        body = [_ResidualGroupParams(n_feats, 3, reduction, n_resblocks) for _ in range(n_resgroups)]
        body.append(default_conv(n_feats, n_feats, 3))
        up = []
        for _ in range(int(math.log(scaling_factor, 2))):
            up += [default_conv(n_feats, 4 * n_feats, 3), nn.PixelShuffle(2)]
        tail = [nn.Sequential(*up), default_conv(n_feats, out_channels, 3)]
        self.head = nn.Sequential(*head)
        self.body = nn.Sequential(*body)
        self.tail = nn.Sequential(*tail)
        self.srcnn = _SRCNNParams(in_channels=3, out_channels=out_channels)

    # the reference's tolerant loader (rcan.py:189-217), kept verbatim in behaviour
    def load_state_dict(self, state_dict: dict, strict: bool = False) -> None:
        own_state = self.state_dict()
        for name, param in state_dict.items():
            if name in own_state:
                if isinstance(param, nn.Parameter):
                    param = param.data
                try:
                    own_state[name].copy_(param)
                except Exception:
                    if name.find("tail") >= 0:
                        logging.info("Replace pre-trained upsampler to new one...")
                    else:
                        raise RuntimeError(f"While copying the parameter named {name}, whose dimensions in the model are {own_state[name].size()} and "
                                           f"whose dimensions in the checkpoint are {param.size()}.")
            elif strict:
                if name.find("tail") == -1:
                    raise KeyError(f'unexpected key "{name}" in state_dict')
        if strict:
            missing = set(own_state.keys()) - set(state_dict.keys())
            if len(missing) > 0:
                raise KeyError(f'missing keys in state_dict: "{missing}"')

    def _conv(self, inp: Tensor, conv: nn.Conv2d, act: str = "none", res1=None, out_mode: str = "nhwc", train: bool = False) -> Tensor:
        # training packs in every conv call: fused optimizers update the weights without bumping their version counters
        scratch, pre, _ = self._layer_pack(conv, force=train)
        return ops.conv2d_nhwc(inp, f32(conv.weight), f32(conv.bias), act=act, res1=res1, out_mode=out_mode, scratch=scratch, prepacked=pre)

    def _conv_t(self, g: Tensor, conv: nn.Conv2d, res1=None, res2=None, gate=None) -> Tensor:
        """Input gradient of ``conv`` (+ res1 + res2, then * ReLU'(gate)), packed transposed on every call."""
        scratch, _, _ = self._layer_pack(conv, transposed=True, force=True)
        return ops.conv2d_nhwc(g, f32(conv.weight), None, transposed=True, res1=res1, res2=res2, gate=gate,
                               gate_neg=0.0, scratch=scratch)

    # ------------------------------------------------------------------ forward (rcan.py:175-186)
    def forward(self, x: Tensor, elev: Tensor, mask: Tensor) -> Tensor:
        check_generator_inputs(x, elev, mask, self.in_channels, "RCAN", "RCAN")
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters())):
            if not self.training:
                raise CsrError("climsr_b200 RCAN trains in train() mode only (eval() mode runs the inference path): call .train() "
                               "before the training forward, or run inference under torch.no_grad() / with frozen parameters")
            return _RCANFunction.apply(self, x, elev, mask, *self.parameters())
        return self._run(x, elev, mask)

    def _run(self, x: Tensor, elev: Tensor, mask: Tensor, saved: Optional[dict] = None) -> Tensor:
        """The forward launch sequence.  saved (training): filled with the activations the backward reads, every RCAB with its own
        pooled sums; the weights are packed in every conv call."""
        n, _, h, w = x.shape
        dev = x.device
        train = saved is not None
        with torch.cuda.device(dev):
            a = ops.nchw_to_nhwc_bf16(x.detach(), 64)
            head = self._conv(a, self.head[0], train=train)                      # x = self.head(x)
            cur = head
            pooled = None if train else torch.empty((n, 64), dtype=torch.float32, device=dev)
            blocks, groups = [], []
            for grp in list(self.body)[:-1]:                                     # ResidualGroup (rcan.py:104-134)
                g_in = cur
                for blk in list(grp.body)[:-1]:                                  # RCAB (rcan.py:71-101)
                    t = self._conv(cur, blk.body[0], act="relu", train=train)
                    r = self._conv(t, blk.body[2], train=train)
                    ca = blk.body[3].conv_du
                    out = torch.empty_like(r)
                    if train:
                        pooled = torch.empty((n, 64), dtype=torch.float32, device=dev)
                        blocks.append((cur, t, r, pooled))
                    check(lib.csr_channel_attention(r.data_ptr(), cur.data_ptr(), f32(ca[0].weight).data_ptr(), f32(ca[0].bias).data_ptr(),
                                                    f32(ca[2].weight).data_ptr(), f32(ca[2].bias).data_ptr(), out.data_ptr(), pooled.data_ptr(),
                                                    n, h, w, 64, ca[0].out_channels, current_stream_ptr()), "csr_channel_attention")
                    cur = out
                groups.append(cur)
                cur = self._conv(cur, grp.body[-1], res1=g_in, train=train)      # res = body(x); res += x
            body_in = cur
            res = self._conv(cur, self.body[-1], res1=head, train=train)         # res = self.body(x); res += x
            up = self.tail[0]
            t, hh, ww = res, h, w
            up_in = []
            for i in range(0, len(up), 2):                                       # Upsampler: conv 64 -> 256, PixelShuffle(2)
                up_in.append(t)
                y4 = self._conv(t, up[i], train=train)
                t = torch.empty((n, 2 * hh, 2 * ww, 64), dtype=torch.bfloat16, device=dev)
                check(lib.csr_pixel_shuffle2(y4.data_ptr(), t.data_ptr(), n, hh, ww, 64, current_stream_ptr()), "csr_pixel_shuffle2")
                hh, ww = 2 * hh, 2 * ww
            y = self._conv(t, self.tail[1], out_mode="f32_planar", train=train)  # (N,1,H,W) fp32
            # x = self.srcnn(torch.cat([x, elev, mask], 1))   (srcnn.py:13-18)
            cat = torch.cat([y, elev.detach().to(dev).float(), mask.detach().to(dev).float()], 1).contiguous()
            s_in = ops.nchw_to_nhwc_bf16(cat, 64)
            s1 = self._conv(s_in, self.srcnn.conv1, act="relu", train=train)
            s2 = self._conv(s1, self.srcnn.conv2, act="relu", train=train)
            if train:
                saved.update(n=n, h=h, w=w, a=a, head=head, blocks=blocks, groups=groups, body_in=body_in, up_in=up_in, tail_in=t,
                             s_in=s_in, s1=s1, s2=s2)
            return self._conv(s2, self.srcnn.conv3, out_mode="f32_planar", train=train)

    # ------------------------------------------------------------------ backward (autograd of rcan.py:175-186)
    def _backward(self, sv: dict, grad_out: Tensor) -> list:
        """Gradients of every parameter, in ``parameters()`` order, as views of one zeroed fp32 buffer."""
        dev = grad_out.device
        n, h, w = sv["n"], sv["h"], sv["w"]
        params = list(self.parameters())
        _, grads = flat_grad_views(params, dev)
        views = dict(zip(params, grads))

        def wgrad(x, g, conv):
            ops.conv2d_wgrad(x, g, tuple(conv.weight.shape), dw=views[conv.weight], db=views[conv.bias])

        with torch.cuda.device(dev):
            g = ops.nchw_to_nhwc_bf16(grad_out.detach().contiguous().float(), 64)
            # SRCNN tail: conv3 <- relu(conv2) <- relu(conv1) <- cat([y, elev, mask])
            sr = self.srcnn
            wgrad(sv["s2"], g, sr.conv3)
            g = self._conv_t(g, sr.conv3, gate=sv["s2"])
            wgrad(sv["s1"], g, sr.conv2)
            g = self._conv_t(g, sr.conv2, gate=sv["s1"])
            wgrad(sv["s_in"], g, sr.conv1)
            g = self._conv_t(g, sr.conv1)                                # channel 0: dL/dy (1, 2: elev / mask, unused)
            # Upsampler: tail.1 <- PixelShuffle <- tail.0.2 <- PixelShuffle <- tail.0.0
            wgrad(sv["tail_in"], g, self.tail[1])
            g = self._conv_t(g, self.tail[1])
            up = self.tail[0]
            for i, t in zip(range(len(up) - 2, -1, -2), reversed(sv["up_in"])):
                hh, ww = t.shape[1], t.shape[2]
                g4 = torch.empty((n, hh, ww, 256), dtype=torch.bfloat16, device=dev)
                check(lib.csr_pixel_unshuffle2(g.data_ptr(), g4.data_ptr(), n, hh, ww, 64, current_stream_ptr()), "csr_pixel_unshuffle2")
                wgrad(t, g4, up[i])
                g = self._conv_t(g4, up[i])
            # body: res = body(head) + head; each group: out = conv(RCABs(g_in)) + g_in; each RCAB: out = CA(res) + cur
            d_res = g
            wgrad(sv["body_in"], d_res, self.body[-1])
            g = self._conv_t(d_res, self.body[-1])
            blocks = iter(reversed(sv["blocks"]))
            scratch = torch.empty(max(lib.csr_channel_attention_backward_scratch_bytes(n, 64), 16), dtype=torch.uint8, device=dev)
            for grp, grp_last_in in zip(reversed(list(self.body)[:-1]), reversed(sv["groups"])):
                d_out = g                                                  # gradient at the group output = at its input (skip)
                wgrad(grp_last_in, d_out, grp.body[-1])
                rcabs = list(grp.body)[:-1]
                if not rcabs:
                    g = self._conv_t(d_out, grp.body[-1], res1=d_out)
                    continue
                g = self._conv_t(d_out, grp.body[-1])
                for k in range(len(rcabs) - 1, -1, -1):
                    blk = rcabs[k]
                    cur, t, r, pooled = next(blocks)
                    ca = blk.body[3].conv_du
                    dr = torch.empty_like(r)
                    check(lib.csr_channel_attention_backward(g.data_ptr(), r.data_ptr(), pooled.data_ptr(), f32(ca[0].weight).data_ptr(),
                                                             f32(ca[0].bias).data_ptr(), f32(ca[2].weight).data_ptr(), f32(ca[2].bias).data_ptr(),
                                                             dr.data_ptr(), views[ca[0].weight].data_ptr(), views[ca[0].bias].data_ptr(),
                                                             views[ca[2].weight].data_ptr(), views[ca[2].bias].data_ptr(), scratch.data_ptr(),
                                                             scratch.numel(), n, h, w, 64, ca[0].out_channels, current_stream_ptr()),
                          "csr_channel_attention_backward")
                    wgrad(t, dr, blk.body[2])
                    dt = self._conv_t(dr, blk.body[2], gate=t)
                    wgrad(cur, dt, blk.body[0])
                    # RCAB skip (+ the group skip at the group's first block)
                    g = self._conv_t(dt, blk.body[0], res1=g, res2=d_out if k == 0 else None)
            # dL/dhead = g + d_res (body skip): the weight gradient is linear in it - two accumulating calls instead of an add pass
            wgrad(sv["a"], g, self.head[0])
            wgrad(sv["a"], d_res, self.head[0])
        return grads


class _RCANFunction(torch.autograd.Function):
    """Training forward / backward of RCAN on the sm_100a kernels.  The saved activations live on this node (``ctx.saved``) and
    are released by its backward or with the graph."""

    @staticmethod
    def forward(ctx, module, x, elev, mask, *params):
        saved = {}
        out = module._run(x, elev, mask, saved)
        ctx.module, ctx.saved = module, saved
        ctx.set_materialize_grads(False)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        n_in = 4 + len(list(ctx.module.parameters()))
        if grad_out is None:
            return (None,) * n_in
        if ctx.needs_input_grad[1]:
            raise CsrError("climsr_b200: the generator does not produce a gradient for its input x (it is data in the reference's "
                           "training loop, climsr/task/pl_generator_pre_training.py:18-33); detach x or clear requires_grad")
        if ctx.saved is None:
            raise CsrError("RCAN's saved activations were released by its first backward; a second backward through the same forward "
                           "(retain_graph=True) is not supported - run the forward again")
        grads = ctx.module._backward(ctx.saved, grad_out)
        ctx.saved = None
        return (None, None, None, None) + tuple(grads)
