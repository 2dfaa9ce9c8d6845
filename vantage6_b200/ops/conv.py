"""Convolution on the hand-written tcgen05 implicit-GEMM kernels (csrc/igemm.cu).

Three entry points, all on NHWC bf16 activations and ``[Cout, R, S, Cin]`` bf16 filters (a PyTorch
``channels_last`` tensor *is* that memory layout, so no conversion happens anywhere):

* :func:`conv_fprop`  -- ``y = conv(x, w)``; with ``bn=...`` the BatchNorm batch statistics of ``y`` (mean, rstd, the
  fused scale/bias, the running-stat update) come out of the same launch, so the separate statistics pass over ``y``
  disappears (ops/bn.py then only runs the apply pass),
* :func:`conv_dgrad`  -- ``dx = conv_transpose(dy, w)`` (stride 1; the filter is read in place through an MN-major
  UMMA descriptor, no transposed / flipped copy),
* :func:`conv_wgrad`  -- ``dw += dy^T . im2col(x)`` accumulated in fp32 **directly into the flat gradient buffer**
  (split-K over pixels, ``red.global.add.v4.f32``), so the bf16 gradient + gradient-sink round trip disappears.

``TcConv2d`` packages them as an autograd function; ``supported()`` says which layer shapes the kernels take
(Cin, Cout multiples of 64, square filter, stride-1 data gradient) -- everything in ResNet-50 except the 16-channel
space-to-depth stem and the data gradient of the six stride-2 layers.

Reference parity: the reference has no compute (SURVEY.md 2.6); the contract is BASELINE.json config 2.
"""
from __future__ import annotations

import os
from typing import Optional, Tuple

import torch

from . import count, native, stream_ptr

_scratch: dict = {}


def igemm_scratch(device) -> torch.Tensor:
    """Counters + per-CTA statistics partials of the FPROP statistics epilogue (zeroed once; the counters reset
    themselves; launches are stream-ordered)."""
    key = str(device)
    buf = _scratch.get(key)
    if buf is None:
        buf = _scratch[key] = torch.zeros(int(native().IGEMM_SCRATCH_FLOATS), device=device, dtype=torch.float32)
    return buf


def _nhwc(x: torch.Tensor) -> Tuple[int, int, int, int]:
    n, c, h, w = x.shape
    return n, h, w, c


def _is_cl(x: torch.Tensor) -> bool:
    return x.dim() == 4 and x.is_contiguous(memory_format=torch.channels_last)


def supported(cin: int, cout: int, r: int, s: int, stride: int, pad: int) -> bool:
    """Layer shapes the tcgen05 kernels take (forward + filter gradient; the data gradient additionally needs stride 1)."""
    return cin % 64 == 0 and cout % 64 == 0 and r == s and stride in (1, 2) and 0 <= pad < r


def dgrad_supported(cin: int, cout: int, r: int, s: int, stride: int, pad: int, h: int = 0, w: int = 0) -> bool:
    if not supported(cin, cout, r, s, stride, pad):
        return False
    return stride == 1 or ((r, pad) in ((3, 1), (1, 0)) and h % 2 == 0 and w % 2 == 0)


def out_size(h: int, r: int, stride: int, pad: int) -> int:
    return (h + 2 * pad - r) // stride + 1


def conv_fprop(x: torch.Tensor, w: torch.Tensor, stride: int = 1, pad: int = 0, bn: Optional[dict] = None,
               bias: Optional[torch.Tensor] = None, act: int = 0, force_im2col: bool = False) -> torch.Tensor:
    """``x``: [N, Cin, H, W] channels_last bf16; ``w``: [Cout, Cin, R, S] channels_last bf16 -> y channels_last bf16.

    ``bn``: dict(gamma, beta, running_mean, running_var, num_batches_tracked, mean, rstd, scale_bias, eps, momentum);
    mean / rstd / scale_bias ([2*Cout]) are outputs."""
    assert x.is_cuda and x.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and _is_cl(x) and _is_cl(w)
    n, h, wd, cin = _nhwc(x)
    cout, cin2, r, s = w.shape
    assert cin == cin2
    p, q = out_size(h, r, stride, pad), out_size(wd, s, stride, pad)
    y = torch.empty((n, cout, p, q), device=x.device, dtype=torch.bfloat16, memory_format=torch.channels_last)
    g = bn or {}

    def ptr(t):
        return 0 if t is None else t.data_ptr()

    count(1)
    native().conv_fprop(x.data_ptr(), w.data_ptr(), y.data_ptr(), ptr(bias), act, n, h, wd, cin, cout, r, s, stride, pad,
                        ptr(g.get("gamma")), ptr(g.get("beta")), ptr(g.get("running_mean")), ptr(g.get("running_var")),
                        ptr(g.get("num_batches_tracked")), ptr(g.get("mean")), ptr(g.get("rstd")), ptr(g.get("scale_bias")),
                        igemm_scratch(x.device).data_ptr() if bn else 0, float(g.get("eps", 1e-5)), float(g.get("momentum", 0.1)),
                        force_im2col, stream_ptr(), 0, 0, 0)
    return y


def conv_dgrad(dy: torch.Tensor, w: torch.Tensor, in_hw: Tuple[int, int], pad: int = 0, force_im2col: bool = False,
               stride: int = 1, add: Optional[torch.Tensor] = None, add_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Data gradient of a convolution: ``dy`` [N, Cout, P, Q] -> dx [N, Cin, H, W] (channels_last bf16).  stride 2 (3x3 /
    pad 1 and 1x1 / pad 0, even H, W): one launch that walks the 4 output-pixel parity classes, each a stride-1 implicit
    GEMM over dY with the sub-filter that reaches it."""
    assert dy.is_cuda and dy.dtype == torch.bfloat16 and _is_cl(dy) and _is_cl(w)
    n, p, q, cout = _nhwc(dy)
    cout2, cin, r, s = w.shape
    h, wd = in_hw
    assert cout == cout2 and p == out_size(h, r, stride, pad) and q == out_size(wd, s, stride, pad)
    dx = torch.empty((n, cin, h, wd), device=dy.device, dtype=torch.bfloat16, memory_format=torch.channels_last)
    if add is not None:         # gradient arriving at the same tensor through another branch: folded into the epilogue (stride 1)
        assert add.shape == dx.shape and add.dtype == torch.bfloat16 and _is_cl(add) and stride == 1
        # add_mask: 1 bit / element ([pixels, C/8] bytes, ops/bn.py): the branch gradient is ``add`` where the bit is set, else 0
        assert add_mask is None or (add_mask.dtype == torch.uint8 and add_mask.numel() * 8 == add.numel())
    count(1)
    native().conv_dgrad(dy.data_ptr(), w.data_ptr(), dx.data_ptr(), n, h, wd, cin, cout, r, s, stride, pad, force_im2col, stream_ptr(),
                        0 if add is None else add.data_ptr(), 0 if (add is None or add_mask is None) else add_mask.data_ptr())
    return dx


def _wgrad(dy, x, dw, n, h, w, cin, cout, r, s, stride, pad, scale, splits, force_im2col, pitches=(0, 0, 0)) -> None:
    """One WGRAD launch.  When a tile's K is split into several ranges, their partial tiles go to a workspace (allocated here, on
    the current stream) and a second kernel adds them into ``dw`` in one fixed order: the same sum on every run."""
    C = native()
    ws_floats = C.conv_wgrad_workspace(n, h, w, cin, cout, r, s, stride, pad, int(splits))
    ws = torch.empty(ws_floats, device=dw.device, dtype=torch.float32) if ws_floats else None
    count(2 if ws_floats else 1)
    C.conv_wgrad(dy.data_ptr(), x.data_ptr(), dw.data_ptr(), n, h, w, cin, cout, r, s, stride, pad, float(scale), int(splits), force_im2col,
                 stream_ptr(), *pitches, 0 if ws is None else ws.data_ptr(), ws_floats)


def conv_wgrad(dy: torch.Tensor, x: torch.Tensor, dw: torch.Tensor, rs: Tuple[int, int], stride: int = 1, pad: int = 0,
               scale: float = 1.0, splits: int = 0, force_im2col: bool = False) -> torch.Tensor:
    """``dw`` (fp32, memory [Cout, R, S, Cin], e.g. the ``.grad`` view of a flat model) ``+= scale * dy^T . im2col(x)``."""
    assert dy.is_cuda and dy.dtype == torch.bfloat16 and x.dtype == torch.bfloat16 and _is_cl(dy) and _is_cl(x)
    assert dw.dtype == torch.float32
    n, h, wd, cin = _nhwc(x)
    cout = dy.shape[1]
    r, s = rs
    assert dw.numel() == cout * r * s * cin
    _wgrad(dy, x, dw, n, h, wd, cin, cout, r, s, stride, pad, scale, splits, force_im2col)
    return dw


# ------------------------------------------------------------------------------------------------- ResNet stem
def stem_fprop(xs: torch.Tensor, ws: torch.Tensor, bn: Optional[dict] = None) -> torch.Tensor:
    """The 7x7 / stride-2 stem as a 4x4 / stride-1 convolution on the 16-channel space-to-depth image ``xs``
    [N, 16, Hs, Ws] (ops/pool.py) -- on the tensor cores: the 4 horizontally adjacent 16-channel pixels of a filter row are
    64 contiguous bf16 in NHWC memory, so the image is read through an im2col map whose "pixels" are those overlapping
    64-element windows (pixel pitch 32 B): a 4x1 convolution with Cin = 64, K = 4 x 64 = 256.  ``bn``: as in
    :func:`conv_fprop` (the batch statistics of the output from the same launch)."""
    n, c16, hs, wsz = xs.shape
    cout = ws.shape[0]
    assert c16 == 16 and tuple(ws.shape[1:]) == (16, 4, 4) and _is_cl(xs) and _is_cl(ws)
    p, q = hs - 3, wsz - 3
    y = torch.empty((n, cout, p, q), device=xs.device, dtype=torch.bfloat16, memory_format=torch.channels_last)
    g = bn or {}

    def ptr(t):
        return 0 if t is None else t.data_ptr()

    count(1)
    native().conv_fprop(xs.data_ptr(), ws.data_ptr(), y.data_ptr(), 0, 0, n, hs, q, 64, cout, 4, 1, 1, 0,
                        ptr(g.get("gamma")), ptr(g.get("beta")), ptr(g.get("running_mean")), ptr(g.get("running_var")),
                        ptr(g.get("num_batches_tracked")), ptr(g.get("mean")), ptr(g.get("rstd")), ptr(g.get("scale_bias")),
                        igemm_scratch(xs.device).data_ptr() if bn else 0, float(g.get("eps", 1e-5)), float(g.get("momentum", 0.1)),
                        True, stream_ptr(), 32, wsz * 32, hs * wsz * 32)
    return y


def stem_wgrad(dy: torch.Tensor, xs: torch.Tensor, dws: torch.Tensor) -> torch.Tensor:
    """``dws`` (fp32 [Cout, 4, 4, 16]) += dy^T . im2col(xs) through the same overlapping-window view."""
    n, c16, hs, wsz = xs.shape
    cout = dy.shape[1]
    assert dws.dtype == torch.float32 and dws.numel() == cout * 256
    _wgrad(dy, xs, dws, n, hs, wsz - 3, 64, cout, 4, 1, 1, 0, 1.0, 0, True, (32, wsz * 32, hs * wsz * 32))
    return dws


FORCE_IM2COL = os.environ.get("V6B200_CONV_FORCE_IM2COL") == "1"


# ------------------------------------------------------------------------------------------------- nn.Linear backward
def linear_bwd_supported(n_out: int, k_in: int) -> bool:
    """dX = dY . W (DGRAD form: K = n_out in 64-blocks) and dW += dY^T . X (WGRAD form: columns = k_in in 64-chunks)."""
    return n_out % 64 == 0 and k_in % 64 == 0


def linear_fprop(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, act: int = 0) -> torch.Tensor:
    """``y[M, N] = act(x[M, K] . w[N, K]^T + bias)`` on the implicit-GEMM kernel (a 1x1 convolution over a 1 x M image): its N tile
    is chosen per problem (64 / 128 / 256 columns), which fills the SMs on shapes where the fixed 128x256 tile of ops/gemm.py
    leaves most of them idle."""
    assert x.is_cuda and x.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and x.is_contiguous() and w.is_contiguous()
    m, k = x.shape
    n, k2 = w.shape
    assert k == k2 and k % 64 == 0 and n % 8 == 0
    y = torch.empty((m, n), device=x.device, dtype=torch.bfloat16)
    count(1)
    native().conv_fprop(x.data_ptr(), w.data_ptr(), y.data_ptr(), 0 if bias is None else bias.data_ptr(), int(act), 1, 1, m, k, n, 1, 1, 1, 0,
                        0, 0, 0, 0, 0, 0, 0, 0, 0, 1e-5, 0.1, False, stream_ptr(), 0, 0, 0)
    return y


def linear_dgrad(dy: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
    """``dx[M, K] = dy[M, N] . w[N, K]`` -- the weight is read in place as an MN-major UMMA operand (no transpose)."""
    assert dy.is_cuda and dy.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and dy.is_contiguous() and w.is_contiguous()
    m, n = dy.shape
    n2, k = w.shape
    assert n == n2
    dx = torch.empty((m, k), device=dy.device, dtype=torch.bfloat16)
    count(1)
    native().conv_dgrad(dy.data_ptr(), w.data_ptr(), dx.data_ptr(), 1, 1, m, k, n, 1, 1, 1, 0, False, stream_ptr(), 0, 0)
    return dx


def linear_wgrad(dy: torch.Tensor, x: torch.Tensor, dw: torch.Tensor, scale: float = 1.0) -> torch.Tensor:
    """``dw[N, K] (fp32) += scale * dy[M, N]^T . x[M, K]`` -- both operands MN-major, split-K over the M rows, fp32
    accumulation straight into ``dw`` (e.g. the ``.grad`` view of a flat model)."""
    assert dy.is_cuda and dy.dtype == torch.bfloat16 and x.dtype == torch.bfloat16 and dy.is_contiguous() and x.is_contiguous()
    assert dw.dtype == torch.float32 and dw.is_contiguous()
    m, n = dy.shape
    m2, k = x.shape
    assert m == m2 and dw.numel() == n * k
    _wgrad(dy, x, dw, 1, 1, m, k, n, 1, 1, 1, 0, scale, 0, False)
    return dw
