"""Convolution with an fp32 master filter and a bf16 compute copy (ResNet-50 local step).

Default path (``V6B200_CONV=tc``): the hand-written tcgen05 implicit-GEMM kernels of csrc/igemm.cu through ops/conv.py --
forward (optionally with the BatchNorm batch statistics of the output in its epilogue), data gradient (filter read in
place through an MN-major descriptor, residual-branch gradient folded into the epilogue: ``GradFork``) and filter gradient
(split-K, fp32 accumulation straight into the flat gradient buffer, issued on a second stream so that it overlaps the
BatchNorm backward passes of the next layer: ``side_wgrad``).

Library arm (``V6B200_CONV=cudnn``, also the fallback for shapes the kernels do not take): ``aten::convolution`` on the
bf16 shadow filter.  What this layer removes there is everything *around* the convolution that the autocast path
launches per layer and per step (profiles/launches_resnet50_fusedbn_v2_r1.txt):

* the fp32 -> bf16 filter cast: the forward reads the bf16 shadow copy that the fused optimizer (K7)
  and the aggregation kernel (K2) keep up to date,
* the NCHW -> NHWC filter conversion: filters live channels-last inside the flat buffers
  (models/flat.py),
* the bf16 -> fp32 gradient cast and the gradient accumulation: the bf16 filter gradient is queued on
  the flat model's gradient sink and added into the flat fp32 gradient buffer by ONE multi-tensor
  kernel per step (ops/optim.py::multi_accumulate).

Without a shadow (CPU tests, the stock-optimizer baseline arm) it is a plain ``nn.Conv2d``.
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import torch
from torch import nn


class _ShadowConvFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, w_bf16, stride, padding, sink, offset):
        y = torch.ops.aten.convolution(x, w_bf16, None, stride, padding, (1, 1), False, (0, 0), 1)
        ctx.save_for_backward(x, w_bf16)
        ctx.conf = (stride, padding)
        ctx.sink, ctx.offset = sink, offset
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w_bf16 = ctx.saved_tensors
        stride, padding = ctx.conf
        dx, dw, _ = torch.ops.aten.convolution_backward(dy, x, w_bf16, None, stride, padding, (1, 1), False, (0, 0), 1,
                                                        (ctx.needs_input_grad[0], True, False))
        if not dw.is_contiguous(memory_format=torch.channels_last):
            dw = dw.contiguous(memory_format=torch.channels_last)
        ctx.sink.append((dw, ctx.offset))        # flushed by FlatModel.flush_grad_sink() after backward
        return dx, None, None, None, None, None, None


def _tc_mode() -> str:
    """V6B200_CONV = tc (default: the hand-written tcgen05 implicit-GEMM kernels, csrc/igemm.cu) | cudnn (library arm)."""
    import os

    return os.environ.get("V6B200_CONV", "tc")


class _SideWgrad:
    """Filter gradients on a second stream.  In the backward pass the data-gradient chain (dgrad -> BatchNorm backward ->
    dgrad ...) is the critical path; the filter gradient of a layer only feeds the optimizer at the end of the step.  Both
    convolution kernels own a whole SM (~200 KB of shared memory per CTA), but the memory-bound BatchNorm backward passes
    of the next layer fit next to a filter-gradient CTA -- so the filter gradients are issued on a side stream (forked
    after ``dy`` exists, joined once by :func:`join_side_wgrad` before the optimizer) and overlap them.  Under CUDA-graph
    capture the fork / join events become graph edges.  Enabled by the trainer (``side_wgrad(True)``); tensors the side
    stream reads are kept referenced until the join, so the caching allocator cannot hand their blocks out early."""

    def __init__(self):
        self.enabled = False
        self.streams: dict = {}
        self.pending: list = []
        self.forked = False

    def stream(self, device) -> "torch.cuda.Stream":
        key = torch.device(device).index
        st = self.streams.get(key)
        if st is None:
            st = self.streams[key] = torch.cuda.Stream(device=device)
        return st


_side = _SideWgrad()


def side_wgrad(enable: bool) -> bool:
    """Switch the side-stream filter gradients on / off (``V6B200_WGRAD_STREAM=0`` keeps them off); returns the state."""
    import os

    _side.enabled = bool(enable) and os.environ.get("V6B200_WGRAD_STREAM", "1") != "0"
    return _side.enabled


def join_side_wgrad() -> None:
    """Make the current stream wait for the filter gradients issued since the last join (call before reading ``.grad``)."""
    if _side.forked:
        for st in _side.streams.values():
            torch.cuda.current_stream(st.device).wait_stream(st)
        _side.forked = False
    _side.pending.clear()


class GradFork:
    """Hand-over of a gradient between the two autograd nodes that consume the SAME tensor at a residual fork (the
    block input feeds conv1 and the identity / downsample branch).  The branch that runs first in the backward pass
    (``producer``) parks its gradient here and returns ``None`` to autograd; the first convolution's data-gradient
    kernel -- always the last consumer to run -- adds it in its epilogue.  One full-tensor add pass per residual block
    disappears (4 % of a ResNet-50 round, profiles/launches_resnet50_v4_r1.txt)."""

    __slots__ = ("grad", "mask", "armed")

    def __init__(self):
        # mask: the parked gradient counts only where this 1-bit-per-element ReLU mask is set (ops/bn.py parks the
        # block-output gradient + the mask instead of writing a masked copy)
        self.grad, self.mask, self.armed = None, None, False


def expand_relu_mask(mask: torch.Tensor, like: torch.Tensor) -> torch.Tensor:
    """[pixels, C/8] mask bytes -> a 0/1 tensor shaped like the channels_last activation ``like`` (fallback paths only)."""
    n, c, h, w = like.shape
    bits = (mask.view(n, h, w, c // 8, 1) >> torch.arange(8, device=mask.device, dtype=torch.uint8)) & 1
    return bits.view(n, h, w, c).permute(0, 3, 1, 2).to(like.dtype)


class _TcConvFn(torch.autograd.Function):
    """Convolution on the hand-written tcgen05 kernels (ops/conv.py): forward = implicit GEMM through TMA im2col maps
    (+ the BatchNorm statistics of the output when ``bn`` is given), data gradient = the same kernel reading the filter
    in place through an MN-major descriptor, filter gradient = split-K implicit GEMM accumulating in fp32 straight into
    ``weight.grad`` (the flat gradient buffer) -- no bf16 gradient tensor, no gradient sink entry."""

    @staticmethod
    def forward(ctx, x, weight, w_bf16, stride, pad, bn, fork_in=None, fork_out=None):
        from ..ops import conv as C

        y = C.conv_fprop(x, w_bf16, stride, pad, bn=bn)
        ctx.save_for_backward(x, w_bf16)
        ctx.conf = (stride, pad)
        ctx.weight = weight
        ctx.fork_in, ctx.fork_out = fork_in, fork_out
        if fork_in is not None and stride == 1:
            fork_in.armed = True            # this node will fold the parked gradient into its data-gradient epilogue
        return y

    @staticmethod
    def backward(ctx, dy):
        from ..ops import conv as C

        x, w_bf16 = ctx.saved_tensors
        stride, pad = ctx.conf
        weight = ctx.weight
        if not dy.is_contiguous(memory_format=torch.channels_last):
            dy = dy.contiguous(memory_format=torch.channels_last)
        cout, cin, r, s = w_bf16.shape
        dx = None
        if ctx.needs_input_grad[0]:
            add = add_mask = None
            if ctx.fork_in is not None and ctx.fork_in.armed:
                add, add_mask = ctx.fork_in.grad, ctx.fork_in.mask
                ctx.fork_in.grad = ctx.fork_in.mask = None
            if C.dgrad_supported(cin, cout, r, s, stride, pad, x.shape[2], x.shape[3]):
                dx = C.conv_dgrad(dy, w_bf16, (x.shape[2], x.shape[3]), pad, stride=stride, add=add, add_mask=add_mask)
                add = None
            else:       # odd spatial sizes under stride 2: library kernel
                dx = torch.ops.aten.convolution_backward(dy, x, w_bf16, None, (stride, stride), (pad, pad), (1, 1), False, (0, 0), 1,
                                                         (True, False, False))[0]
            if add is not None:
                dx = dx + (add if add_mask is None else add * expand_relu_mask(add_mask, add))
            if ctx.fork_out is not None and ctx.fork_out.armed:      # downsample branch: park, the block's conv1 adds it
                ctx.fork_out.grad, ctx.fork_out.mask, dx = dx, None, None
        g = weight.grad
        direct = (g is not None and g.dtype == torch.float32 and g.shape == weight.shape
                  and g.is_contiguous(memory_format=torch.channels_last))
        if direct:
            if _side.enabled:
                st = _side.stream(x.device)
                st.wait_stream(torch.cuda.current_stream(x.device))      # dy exists, the gradient buffer is zeroed
                with torch.cuda.stream(st):
                    C.conv_wgrad(dy, x, g, (r, s), stride, pad)
                _side.pending.append((dy, x))
                _side.forked = True
            else:
                C.conv_wgrad(dy, x, g, (r, s), stride, pad)
            return dx, None, None, None, None, None, None, None
        dw = torch.zeros((cout, r, s, cin), device=x.device, dtype=torch.float32)
        C.conv_wgrad(dy, x, dw, (r, s), stride, pad)
        return dx, dw.permute(0, 3, 1, 2), None, None, None, None, None, None


class ShadowConv2d(nn.Conv2d):
    """``nn.Conv2d`` (no bias, groups=1, dilation=1) whose forward uses the bf16 shadow filter when attached."""

    def __init__(self, *args, **kw):
        super().__init__(*args, **kw)
        assert self.bias is None and self.groups == 1 and tuple(self.dilation) == (1, 1) and self.padding_mode == "zeros"
        self.w_bf16: Optional[torch.Tensor] = None        # channels-last view into the bf16 shadow buffer
        self._sink: Optional[List[Tuple[torch.Tensor, int]]] = None
        self._offset = 0

    def attach(self, w_bf16: torch.Tensor, sink: list, offset: int) -> None:
        self.w_bf16, self._sink, self._offset = w_bf16, sink, int(offset)

    def tc_supported(self, x: torch.Tensor) -> bool:
        from ..ops import conv as C

        return (_tc_mode() == "tc" and self.w_bf16 is not None and x.is_cuda and x.dim() == 4
                and self.stride[0] == self.stride[1] and self.padding[0] == self.padding[1]
                and C.supported(self.in_channels, self.out_channels, self.kernel_size[0], self.kernel_size[1], self.stride[0],
                                self.padding[0])
                and x.is_contiguous(memory_format=torch.channels_last))

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if self.w_bf16 is None or not x.is_cuda or not torch.is_grad_enabled() or not self.weight.requires_grad:
            if self.w_bf16 is not None and x.is_cuda:
                return torch.ops.aten.convolution(x.to(torch.bfloat16), self.w_bf16, None, self.stride, self.padding, (1, 1),
                                                  False, (0, 0), 1)
            return super().forward(x)
        if x.dtype != torch.bfloat16:
            x = x.to(torch.bfloat16)
        if self.tc_supported(x):
            return _TcConvFn.apply(x, self.weight, self.w_bf16, self.stride[0], self.padding[0], None)
        return _ShadowConvFn.apply(x, self.weight, self.w_bf16, tuple(self.stride), tuple(self.padding), self._sink,
                                   self._offset)


def conv_bn(conv: nn.Module, bn: nn.Module, x: torch.Tensor, residual: Optional[torch.Tensor] = None,
            fork_in: Optional[GradFork] = None, fork_out: Optional[GradFork] = None, res_fork: Optional[GradFork] = None) -> torch.Tensor:
    """``bn(conv(x), residual)``.  On the tcgen05 path the BatchNorm batch statistics come out of the convolution's
    epilogue (one launch less and one full read of the activation less per layer); everywhere else the two modules are
    simply composed.  ``fork_in`` / ``fork_out`` / ``res_fork``: see :class:`GradFork` (``fork_in``: this convolution's
    data gradient absorbs the parked gradient; ``fork_out``: this convolution parks its data gradient; ``res_fork``: the
    BatchNorm parks the gradient of its residual input)."""
    from ..ops.bn import FusedBatchNormAct

    if (isinstance(conv, ShadowConv2d) and isinstance(bn, FusedBatchNormAct) and bn.training and torch.is_grad_enabled()
            and conv.w_bf16 is not None and conv.weight.requires_grad and x.is_cuda):
        if x.dtype != torch.bfloat16:
            x = x.to(torch.bfloat16)
        if conv.tc_supported(x) and (residual is None or residual.is_contiguous(memory_format=torch.channels_last)):
            stats = bn.stats_buffers(x.device)
            y = _TcConvFn.apply(x, conv.weight, conv.w_bf16, conv.stride[0], conv.padding[0], stats, fork_in, fork_out)
            return bn.apply_pre(y, stats, residual, res_fork=res_fork)
    return bn(conv(x), residual=residual) if residual is not None else bn(conv(x))
