"""Single-op wrappers over the C-ABI (used by parity tests and as building blocks)."""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch
from torch import Tensor

from ._lib import ConvDesc, WgradDesc, check, current_stream_ptr, lib

ACT = {"none": 0, "lrelu": 1, "relu": 2, "lrelu_slope": 4}
OUT_MODE = {"nhwc": 0, "f32_planar": 2, "f32_nhwc": 3, "split": 4}


def nchw_to_nhwc_bf16(x: Tensor, dst_c: int = 64) -> Tensor:
    """fp32 NCHW (c <= 16) -> bf16 NHWC with dst_c channels per pixel (channels >= c are zero)."""
    n, c, h, w = x.shape
    out = torch.zeros((n, h, w, dst_c), dtype=torch.bfloat16, device=x.device)
    xs = x.contiguous().float()
    check(lib.csr_nchw_f32_to_nhwc_bf16(xs.data_ptr(), out.data_ptr(), n, c, h, w, dst_c, 16 if dst_c >= 16 else 8,
                                        current_stream_ptr()), "csr_nchw_f32_to_nhwc_bf16")
    return out


def nhwc_bf16_to_nchw(x: Tensor, c: int, coff: int = 0) -> Tensor:
    n, h, w, cc = x.shape
    out = torch.empty((n, c, h, w), dtype=torch.float32, device=x.device)
    check(lib.csr_nhwc_bf16_to_nchw_f32(x.data_ptr(), out.data_ptr(), n, c, h, w, cc, coff, current_stream_ptr()),
          "csr_nhwc_bf16_to_nchw_f32")
    return out


def nchw_to_nhwc_split(x: Tensor, dst_c: int = 16, out: Optional[Tensor] = None) -> Tensor:
    """fp32 NCHW (c <= 3) -> bf16 NHWC hi/lo pairs [hi_0..hi_{c-1}, lo_0..lo_{c-1}, 0...] with dst_c channels per pixel
    (csr_nchw_f32_to_nhwc_split).  ``out``: an (n, h, w, dst_c) bf16 view to write instead of a new buffer."""
    n, c, h, w = x.shape
    if out is None:
        out = torch.empty((n, h, w, dst_c), dtype=torch.bfloat16, device=x.device)
    xs = x.contiguous().float()
    check(lib.csr_nchw_f32_to_nhwc_split(xs.data_ptr(), out.data_ptr(), n, c, h, w, dst_c, current_stream_ptr()),
          "csr_nchw_f32_to_nhwc_split")
    return out


def maxpool2x2_split(x: Tensor) -> Tensor:
    """nn.MaxPool2d(2) of the values hi + lo held by a bf16 NHWC (n, h, w, 2c) hi/lo buffer, re-split (csr_maxpool2x2_split)."""
    n, h, w, c2 = x.shape
    out = torch.empty((n, h // 2, w // 2, c2), dtype=torch.bfloat16, device=x.device)
    check(lib.csr_maxpool2x2_split(x.data_ptr(), out.data_ptr(), n, h, w, c2 // 2, current_stream_ptr()), "csr_maxpool2x2_split")
    return out


def conv2d_nhwc(inp: Tensor, weight: Tensor, bias: Optional[Tensor], *, act: str = "none", out: Optional[Tensor] = None,
                out_coff: int = 0, out_mode: str = "nhwc", in_coff: int = 0, in_up2: bool = False, transposed: bool = False,
                res1: Optional[Tensor] = None, res1_coff: int = 0, scale1: float = 1.0,
                res2: Optional[Tensor] = None, res2_coff: int = 0, scale2: float = 1.0,
                gate: Optional[Tensor] = None, gate_coff: int = 0, gate_from: int = 0, gate_neg: float = 0.2,
                act_slope: float = 0.0, scratch: Optional[Tensor] = None, prepacked: bool = False) -> Tensor:
    """One KxK stride-1 'same' conv on a bf16 NHWC buffer via csr_conv2d_nhwc.

    Reads input channels [in_coff, in_coff+cin); writes act(conv+bias) (then *scale1+res1, *scale2+res2, lrelu-gate) into
    channels [out_coff, out_coff+cout) of `out` (allocated as a 64-channel-padded buffer when None; out_mode "split": hi in
    [out_coff, out_coff+cout), lo in [out_coff+cout, out_coff+2*cout), a 2*cout-channel buffer when None).  in_up2: the input
    is nearest-x2 upsampled first (output is 2h x 2w).  transposed: `weight` is the forward layer's OIHW tensor and the
    op computed is that layer's input gradient (cin/cout swap roles).
    """
    n, h, w, in_c = inp.shape
    if transposed:
        cin, cout, kh, kw = weight.shape
    else:
        cout, cin, kh, kw = weight.shape
    mode = OUT_MODE[out_mode]
    s = 2 if in_up2 else 1
    if out is None:
        if mode == 2:
            out = torch.empty((n, 1, s * h, s * w), dtype=torch.float32, device=inp.device)
        elif mode == 4:
            out = torch.empty((n, h, w, out_coff + 2 * cout), dtype=torch.bfloat16, device=inp.device)
        else:
            oc = (out_coff + cout + 63) // 64 * 64
            # every channel of every pixel is written when the layer fills the buffer exactly: no zero fill needed then
            alloc = torch.empty if (out_coff == 0 and cout == oc) else torch.zeros
            out = alloc((n, s * h, s * w, oc), dtype=torch.float32 if mode == 3 else torch.bfloat16, device=inp.device)
    out_c = 1 if mode == 2 else out.shape[-1]
    d = ConvDesc(n, h, w, cin, cout, kh, kw, in_c, in_coff, out_c, out_coff, ACT[act], mode, int(in_up2), int(transposed),
                 scale1, scale2, res1.shape[-1] if res1 is not None else 0, res1_coff,
                 res2.shape[-1] if res2 is not None else 0, res2_coff,
                 gate.shape[-1] if gate is not None else 0, gate_coff, gate_from, gate_neg, act_slope)
    nbytes = lib.csr_conv2d_scratch_bytes(C.byref(d))
    if scratch is None:
        if prepacked:
            raise ValueError("prepacked=True needs the scratch buffer of the call that packed the weights")
        scratch = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=inp.device)
    elif scratch.numel() < nbytes:
        raise ValueError(f"scratch holds {scratch.numel()} bytes, the layer needs {nbytes}")
    # prepacked: `scratch` already holds this layer's packed weights / bias (same weights, same shape): skip the pack launch
    wc = None if prepacked else weight.contiguous().float()
    bc = bias.contiguous().float() if (bias is not None and not prepacked) else None
    check(lib.csr_conv2d_nhwc(C.byref(d), inp.data_ptr(), wc.data_ptr() if wc is not None else None, bc.data_ptr() if bc is not None else None, out.data_ptr(),
                              res1.data_ptr() if res1 is not None else None, res2.data_ptr() if res2 is not None else None,
                              gate.data_ptr() if gate is not None else None,
                              scratch.data_ptr(), nbytes, current_stream_ptr()), "csr_conv2d_nhwc")
    return out


def conv2d_pack(weight: Tensor, bias: Optional[Tensor], scratch: Tensor, transposed: bool = False) -> None:
    """Pack one layer's weights / bias into ``scratch`` (csr_conv2d_pack) for later ``conv2d_nhwc(..., prepacked=True)`` calls."""
    if transposed:
        cin, cout, kh, kw = weight.shape
    else:
        cout, cin, kh, kw = weight.shape
    d = ConvDesc(1, 8, 8, cin, cout, kh, kw, 64, 0, 64, 0, 0, 0, 0, int(transposed), 1.0, 1.0, 0, 0, 0, 0, 0, 0, 0, 0.2, 0.0)
    wc = weight.detach().contiguous().float()
    bc = bias.detach().contiguous().float() if bias is not None else None
    with torch.cuda.device(weight.device):
        check(lib.csr_conv2d_pack(C.byref(d), wc.data_ptr(), bc.data_ptr() if bc is not None else None, scratch.data_ptr(), scratch.numel(),
                                  current_stream_ptr()), "csr_conv2d_pack")


def conv2d_scratch_bytes(cout: int, cin: int, kh: int, kw: int, transposed: bool = False) -> int:
    """Bytes of packed weights + bias of one layer (shape-only query)."""
    d = ConvDesc(1, 8, 8, cin, cout, kh, kw, 64, 0, 64, 0, 0, 0, 0, int(transposed), 1.0, 1.0, 0, 0, 0, 0, 0, 0, 0, 0.2, 0.0)
    return int(lib.csr_conv2d_scratch_bytes(C.byref(d)))


def conv2d_wgrad(x: Tensor, g: Tensor, weight_shape, *, x_coff: int = 0, g_coff: int = 0, in_up2: bool = False, scale: float = 1.0,
                 dw: Optional[Tensor] = None, db: Optional[Tensor] = None, want_bias: bool = True):
    """Weight / bias gradient of a KxK 'same' conv: x (n,h,w,Cx) bf16 input, g (n,h,w,Cg) bf16 output gradient
    (2h x 2w when in_up2).  Accumulates into dw (cout,cin,kh,kw) / db (cout) fp32 (allocated zeroed when None)."""
    n, h, w, x_c = x.shape
    cout, cin, kh, kw = weight_shape
    if dw is None:
        dw = torch.zeros(weight_shape, dtype=torch.float32, device=x.device)
    if db is None and want_bias:
        db = torch.zeros((cout,), dtype=torch.float32, device=x.device)
    d = WgradDesc(n, h, w, cin, cout, kh, kw, x_c, x_coff, g.shape[-1], g_coff, int(in_up2), scale)
    nbytes = lib.csr_conv2d_wgrad_scratch_bytes(C.byref(d))
    scratch = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=x.device)
    check(lib.csr_conv2d_wgrad(C.byref(d), x.data_ptr(), g.data_ptr(), dw.data_ptr(), db.data_ptr() if db is not None else None,
                               scratch.data_ptr(), nbytes, current_stream_ptr()), "csr_conv2d_wgrad")
    return dw, db
