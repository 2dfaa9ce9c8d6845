"""ResNet-50 (BASELINE config 2: "ResNet-50 FedAvg, 8 GPU-nodes, 1 local epoch/round, synthetic
ImageNet-shape").  Standard bottleneck architecture (v1.5: stride on the 3x3), 25.6 M
parameters = 102 MB fp32 -- the payload of the broadcast / reduction rooflines in BASELINE.md.

Convolutions run on cuDNN (library code, models/conv.py); what is hand-written for this model is
everything around them: fused BatchNorm(+add)(+ReLU) (ops/bn.py), the bf16-shadow / gradient-sink
plumbing that removes the per-layer cast / layout / accumulate launches, the fused flat SGD step (K7),
the FedAvg reduce + server optimizer + broadcast kernel (K2) and the CUDA-graph captured local step.
"""
from __future__ import annotations

import torch
from torch import nn

from .conv import GradFork, ShadowConv2d, conv_bn


class _StockBNAct(nn.BatchNorm2d):
    """Stock path with the same call signature as FusedBatchNormAct (baseline arm / comparisons)."""

    def __init__(self, num_features: int, relu: bool = True):
        super().__init__(num_features)
        self.relu = relu

    def forward(self, x, residual=None, relu=None):
        relu = self.relu if relu is None else relu
        y = super().forward(x)
        if residual is not None:
            y = y + residual
        return torch.relu(y) if relu else y


def _bn(planes: int, relu: bool, fused: bool) -> nn.Module:
    if fused:
        from ..ops.bn import FusedBatchNormAct

        return FusedBatchNormAct(planes, relu=relu)
    return _StockBNAct(planes, relu=relu)


def _maxpool(fused: bool) -> nn.Module:
    if fused:
        from ..ops.pool import MaxPool3x3s2

        return MaxPool3x3s2()
    return nn.MaxPool2d(3, stride=2, padding=1)


class Bottleneck(nn.Module):
    expansion = 4

    def __init__(self, inplanes: int, planes: int, stride: int = 1, downsample: nn.Module | None = None,
                 fused_bn: bool = True):
        super().__init__()
        self.conv1 = ShadowConv2d(inplanes, planes, 1, bias=False)
        self.bn1 = _bn(planes, True, fused_bn)
        self.conv2 = ShadowConv2d(planes, planes, 3, stride=stride, padding=1, bias=False)
        self.bn2 = _bn(planes, True, fused_bn)
        self.conv3 = ShadowConv2d(planes, planes * 4, 1, bias=False)
        self.bn3 = _bn(planes * 4, True, fused_bn)
        self.downsample = downsample

    def forward(self, x):
        # the block input feeds conv1 AND the identity / downsample branch: the gradient of the second branch is handed to
        # conv1's data-gradient kernel instead of being added by a separate pass (GradFork; only armed on the tcgen05 path)
        fork = GradFork() if (self.training and torch.is_grad_enabled() and x.requires_grad) else None
        out = conv_bn(self.conv1, self.bn1, x, fork_in=fork)       # conv (+ BN statistics in its epilogue) -> BN apply + ReLU
        out = conv_bn(self.conv2, self.bn2, out)
        if self.downsample is None:
            return conv_bn(self.conv3, self.bn3, out, residual=x, res_fork=fork)     # BN + residual add + ReLU in one pass
        idt = conv_bn(self.downsample[0], self.downsample[1], x, fork_out=fork)
        return conv_bn(self.conv3, self.bn3, out, residual=idt)


class ResNet(nn.Module):
    def __init__(self, layers=(3, 4, 6, 3), num_classes: int = 1000, width: int = 64, fused_bn: bool = True):
        super().__init__()
        self.inplanes = width
        self.fused_bn = fused_bn
        self.conv1 = ShadowConv2d(3, width, 7, stride=2, padding=3, bias=False)
        self.bn1 = _bn(width, True, fused_bn)
        self.maxpool = _maxpool(fused_bn)
        self.layer1 = self._make_layer(width, layers[0])
        self.layer2 = self._make_layer(width * 2, layers[1], stride=2)
        self.layer3 = self._make_layer(width * 4, layers[2], stride=2)
        self.layer4 = self._make_layer(width * 8, layers[3], stride=2)
        self.avgpool = nn.AdaptiveAvgPool2d((1, 1))
        self.fc = nn.Linear(width * 8 * 4, num_classes)
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")
            elif isinstance(m, nn.BatchNorm2d):
                nn.init.ones_(m.weight)
                nn.init.zeros_(m.bias)
        for m in self.modules():
            if isinstance(m, Bottleneck):
                nn.init.zeros_(m.bn3.weight)       # zero-init last BN of each residual branch

    def _make_layer(self, planes: int, blocks: int, stride: int = 1) -> nn.Sequential:
        downsample = None
        if stride != 1 or self.inplanes != planes * 4:
            downsample = nn.Sequential(ShadowConv2d(self.inplanes, planes * 4, 1, stride=stride, bias=False),
                                       _bn(planes * 4, False, self.fused_bn))
        layers = [Bottleneck(self.inplanes, planes, stride, downsample, self.fused_bn)]
        self.inplanes = planes * 4
        layers += [Bottleneck(self.inplanes, planes, fused_bn=self.fused_bn) for _ in range(1, blocks)]
        return nn.Sequential(*layers)

    def _stem(self, x: torch.Tensor) -> torch.Tensor:
        """conv1 + bn1(+ReLU).  uint8 NCHW images are normalised on the GPU (the host only ships raw bytes);
        on the fused path the stem runs as a space-to-depth 4x4 convolution (ops/pool.py::stem_s2d)."""
        if x.dtype != torch.uint8:
            return self.bn1(self.conv1(x.contiguous(memory_format=torch.channels_last)))
        bf16_stem = torch.is_autocast_enabled() or getattr(self.conv1, "w_bf16", None) is not None
        if self.fused_bn and x.is_cuda and bf16_stem and torch.is_grad_enabled():
            from ..ops import pool

            if pool.stem_s2d_supported(x, self.conv1):
                if self.training and pool.stem_stats_fused(self.conv1) and hasattr(self.bn1, "stats_buffers"):
                    stats = self.bn1.stats_buffers(x.device)        # batch statistics out of the convolution's epilogue
                    y = pool.stem_s2d(x, self.conv1, _MEAN, _STD, bn=stats)
                    return self.bn1.apply_pre(y, stats)
                return self.bn1(pool.stem_s2d(x, self.conv1, _MEAN, _STD))
            if x.is_contiguous() and (x.shape[2] * x.shape[3]) % 4 == 0:
                return self.bn1(self.conv1(pool.image_normalize(x, _MEAN, _STD)))
        key = str(x.device)
        if key not in _NORM_CACHE:      # created on the eager warm-up pass, never during graph capture
            _NORM_CACHE[key] = (torch.tensor(_MEAN, device=x.device, dtype=torch.float32).view(1, 3, 1, 1),
                                1.0 / torch.tensor(_STD, device=x.device, dtype=torch.float32).view(1, 3, 1, 1))
        mean, inv_std = _NORM_CACHE[key]
        x = ((x.float() - mean) * inv_std).contiguous(memory_format=torch.channels_last)
        return self.bn1(self.conv1(x))

    def forward(self, x):
        x = self.maxpool(self._stem(x))
        x = self.layer4(self.layer3(self.layer2(self.layer1(x))))
        return self.fc(torch.flatten(self.avgpool(x), 1))


_MEAN = (0.485 * 255, 0.456 * 255, 0.406 * 255)
_STD = (0.229 * 255, 0.224 * 255, 0.225 * 255)
_NORM_CACHE: dict = {}


def resnet50(num_classes: int = 1000, fused_bn: bool = True) -> ResNet:
    return ResNet((3, 4, 6, 3), num_classes, fused_bn=fused_bn)


def resnet_tiny(num_classes: int = 10, fused_bn: bool = True) -> ResNet:
    """Same code path at toy size (smoke tests, CPU tests)."""
    return ResNet((1, 1, 1, 1), num_classes, width=8, fused_bn=fused_bn)


def imagenet_forward_loss(model: nn.Module, x: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    """uint8 NCHW images (or already-normalised float images) -> logits -> cross-entropy.

    The normalisation runs on the GPU inside the captured step (ResNet._stem), so the host only ever ships the
    raw uint8 batch (9.6 MB for 64x3x224x224) over PCIe.
    """
    return nn.functional.cross_entropy(model(x).float(), y)
