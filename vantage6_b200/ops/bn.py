"""Fused BatchNorm2d (+ residual add) (+ ReLU) for channels-last bf16 activations (csrc/bn.cu).

``FusedBatchNormAct`` is a drop-in ``nn.BatchNorm2d`` subclass (same parameters / buffers / state
dict) whose forward takes the optional residual and fuses the activation:

    y = relu( BN(x) + residual )

On CUDA with channels-last bf16 inputs the hand-written kernels run (training: batch statistics,
running-stat update, saved mean/rstd for the backward; eval: running statistics); anywhere else the
stock PyTorch ops are used (CPU tests, fp32 inputs).
"""
from __future__ import annotations

from typing import Optional

import torch
from torch import nn

from . import count, native, stream_ptr, tree_scratch

_scratch: dict = {}


def _get_scratch(device, C: int):
    """(reduction scratch shared by every BN launch of the device -- partials + self-resetting arrival
    counters, zeroed once --, per-C backward coefficient buffer).  Launches are stream-ordered."""
    key = str(device)
    red = tree_scratch(device)
    coef = _scratch.get((key, C))
    if coef is None:
        coef = _scratch[(key, C)] = torch.empty(3 * C, device=device, dtype=torch.float32)
    return red, coef


def _fast_path(x: torch.Tensor) -> bool:
    if not (x.is_cuda and x.dtype == torch.bfloat16 and x.dim() == 4):
        return False
    C = x.shape[1]
    cg = C // 8
    return C % 8 == 0 and 1 <= cg <= 256 and (cg & (cg - 1)) == 0 and x.is_contiguous(memory_format=torch.channels_last)


class _BNFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, residual, gamma, beta, running_mean, running_var, num_batches_tracked, eps, momentum, relu, pre=None,
                res_fork=None):
        """``pre`` = (mean, rstd, scale_bias) already produced by the convolution that wrote ``x`` (the statistics
        epilogue of csrc/igemm.cu, which also updated the running statistics): only the apply pass runs here."""
        N, C, H, W = x.shape
        R = N * H * W
        y = torch.empty_like(x)                              # preserves channels_last strides
        mask = torch.empty((R, C // 8), device=x.device, dtype=torch.uint8) if relu else None    # 1 bit / element
        if pre is not None:
            mean, rstd, scale_bias = pre
            count(1)
            native().bn_apply(x.data_ptr(), 0 if residual is None else residual.data_ptr(), scale_bias.data_ptr(),
                              scale_bias.data_ptr() + 4 * C, y.data_ptr(), 0 if mask is None else mask.data_ptr(), R, C, relu,
                              stream_ptr())
        else:
            mean = torch.empty(C, device=x.device, dtype=torch.float32)
            rstd = torch.empty(C, device=x.device, dtype=torch.float32)
            scale_bias = torch.empty(2 * C, device=x.device, dtype=torch.float32)
            part, _ = _get_scratch(x.device, C)
            count(2)                                             # stats(+finalize) + apply
            native().bn_fwd(x.data_ptr(), 0 if residual is None else residual.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                            0 if running_mean is None else running_mean.data_ptr(),
                            0 if running_var is None else running_var.data_ptr(),
                            0 if num_batches_tracked is None else num_batches_tracked.data_ptr(), y.data_ptr(),
                            0 if mask is None else mask.data_ptr(), mean.data_ptr(), rstd.data_ptr(),
                            scale_bias.data_ptr(), part.data_ptr(), R, C, eps, momentum, relu, stream_ptr())
        ctx.save_for_backward(x, mask, gamma, mean, rstd)        # the ReLU mask, not y: 16x fewer bytes re-read
        ctx.relu, ctx.has_res, ctx.R, ctx.C = relu, residual is not None, R, C
        ctx.params = (gamma, beta)
        ctx.res_fork = res_fork             # models/conv.py::GradFork: park the residual gradient for the block's first conv
        return y

    @staticmethod
    def backward(ctx, dy):
        x, mask, gamma, mean, rstd = ctx.saved_tensors
        if not dy.is_contiguous(memory_format=torch.channels_last):
            dy = dy.contiguous(memory_format=torch.channels_last)
        dx = torch.empty_like(x)
        # residual branch gradient = dy . relu'(y).  With an armed GradFork (models/conv.py) the block's first convolution
        # folds it into its data-gradient epilogue straight from (dy, mask): no masked copy is written at all
        park = ctx.has_res and ctx.res_fork is not None and ctx.res_fork.armed and (mask is not None or not ctx.relu)
        dres = torch.empty_like(x) if (ctx.has_res and not park) else None
        # Flat-buffer models pre-allocate .grad as views of one fp32 gradient buffer (models/flat.py): the
        # kernel then accumulates dgamma / dbeta straight into it (no AccumulateGrad add launches).
        pg, pb = ctx.params
        direct = all(p.grad is not None and p.grad.dtype == torch.float32 and p.grad.is_contiguous() for p in (pg, pb))
        dgamma = pg.grad if direct else torch.empty_like(gamma)
        dbeta = pb.grad if direct else torch.empty_like(gamma)
        part, coef = _get_scratch(x.device, ctx.C)
        count(2)                                                 # reduce(+finalize) + apply
        native().bn_bwd(dy.data_ptr(), 0 if mask is None else mask.data_ptr(), x.data_ptr(), gamma.data_ptr(), mean.data_ptr(),
                        rstd.data_ptr(), dx.data_ptr(), 0 if dres is None else dres.data_ptr(), dgamma.data_ptr(),
                        dbeta.data_ptr(), coef.data_ptr(), part.data_ptr(), ctx.R, ctx.C, ctx.relu, direct, stream_ptr())
        if park:
            ctx.res_fork.grad, ctx.res_fork.mask = dy, (mask if ctx.relu else None)
        if direct:
            return dx, dres, None, None, None, None, None, None, None, None, None, None
        return dx, dres, dgamma, dbeta, None, None, None, None, None, None, None, None


class FusedBatchNormAct(nn.BatchNorm2d):
    """BatchNorm2d with fused residual add and ReLU (``relu`` is the module default, overridable per call)."""

    def __init__(self, num_features: int, relu: bool = True, **kw):
        super().__init__(num_features, **kw)
        self.relu = relu

    def stats_buffers(self, device) -> dict:
        """Arguments of the statistics epilogue of the producing convolution (ops/conv.py::conv_fprop ``bn=``): the
        layer's affine parameters and running statistics plus fresh per-call outputs (mean, rstd, scale | bias)."""
        C = self.num_features
        return dict(gamma=self.weight, beta=self.bias, running_mean=self.running_mean, running_var=self.running_var,
                    num_batches_tracked=self.num_batches_tracked, mean=torch.empty(C, device=device, dtype=torch.float32),
                    rstd=torch.empty(C, device=device, dtype=torch.float32),
                    scale_bias=torch.empty(2 * C, device=device, dtype=torch.float32), eps=self.eps,
                    momentum=0.1 if self.momentum is None else self.momentum)

    def apply_pre(self, x: torch.Tensor, stats: dict, residual: Optional[torch.Tensor] = None, relu: Optional[bool] = None,
                  res_fork=None):
        """Training forward when the batch statistics of ``x`` were computed by the convolution that produced it."""
        relu = self.relu if relu is None else relu
        return _BNFn.apply(x, residual, self.weight, self.bias, self.running_mean, self.running_var, self.num_batches_tracked,
                           self.eps, stats["momentum"], relu, (stats["mean"], stats["rstd"], stats["scale_bias"]), res_fork)

    def forward(self, x: torch.Tensor, residual: Optional[torch.Tensor] = None, relu: Optional[bool] = None) -> torch.Tensor:
        relu = self.relu if relu is None else relu
        if _fast_path(x) and (residual is None or (_fast_path(residual) and residual.shape == x.shape)):
            mom = 0.1 if self.momentum is None else self.momentum
            if self.training:
                return _BNFn.apply(x, residual, self.weight, self.bias, self.running_mean, self.running_var,
                                   self.num_batches_tracked, self.eps, mom, relu)      # the kernel also bumps the counter
            # eval: per-channel affine from the running statistics, one fused pass
            scale = self.weight.float() * torch.rsqrt(self.running_var + self.eps)
            bias = self.bias.float() - self.running_mean * scale
            y = torch.empty_like(x)
            N, C, H, W = x.shape
            native().bn_apply(x.data_ptr(), 0 if residual is None else residual.data_ptr(), scale.data_ptr(), bias.data_ptr(),
                              y.data_ptr(), 0, N * H * W, C, relu, stream_ptr())
            return y
        y = super().forward(x)
        if residual is not None:
            y = y + residual
        return torch.relu(y) if relu else y
