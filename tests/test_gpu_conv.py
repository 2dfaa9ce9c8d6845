"""tcgen05 implicit-GEMM convolution kernels (csrc/igemm.cu) against fp32 PyTorch references: forward (+ fused BatchNorm
statistics), data gradient, filter gradient, every ResNet-50 layer family (1x1, 3x3, strided, partial tiles), and the
model-level equivalence of the tcgen05 path with the cuDNN path."""
import os

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    from vantage6_b200.ops import native

    native()
    torch.cuda.set_device(0)
    return torch.device("cuda", 0)


def _t(shape, seed, scale=1.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(shape, device="cuda", generator=g) * scale).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)


CASES = [  # n, cin, cout, h, w, k, stride, pad
    (2, 64, 64, 8, 8, 1, 1, 0), (4, 64, 256, 28, 28, 1, 1, 0), (4, 256, 64, 28, 28, 1, 1, 0), (3, 1024, 2048, 7, 7, 1, 1, 0),
    (2, 64, 64, 8, 8, 3, 1, 1), (4, 64, 64, 28, 28, 3, 1, 1), (4, 128, 128, 14, 14, 3, 1, 1), (5, 512, 512, 7, 7, 3, 1, 1),
    (4, 128, 128, 28, 28, 3, 2, 1), (4, 256, 512, 28, 28, 1, 2, 0), (2, 64, 192, 9, 11, 3, 1, 1),
]


@pytest.mark.parametrize("n,cin,cout,h,w,k,stride,pad", CASES)
def test_conv_fprop_matches_fp32_conv2d(dev, n, cin, cout, h, w, k, stride, pad):
    from vantage6_b200.ops import conv as C

    x, wt = _t((n, cin, h, w), 1), _t((cout, cin, k, k), 2, (cin * k * k) ** -0.5)
    y = C.conv_fprop(x, wt, stride, pad)
    ref = F.conv2d(x.float(), wt.float(), stride=stride, padding=pad)
    assert y.shape == ref.shape and y.is_contiguous(memory_format=torch.channels_last)
    torch.testing.assert_close(y.float(), ref, rtol=2e-2, atol=2e-2)


@pytest.mark.parametrize("n,cin,cout,h,w,k,stride,pad", [c for c in CASES if c[2] % 64 == 0][:9])
def test_conv_fprop_batchnorm_statistics_epilogue(dev, n, cin, cout, h, w, k, stride, pad):
    from vantage6_b200.ops import conv as C

    x, wt = _t((n, cin, h, w), 3), _t((cout, cin, k, k), 4, (cin * k * k) ** -0.5)
    bn = dict(gamma=torch.rand(cout, device=dev) + 0.5, beta=torch.randn(cout, device=dev), running_mean=torch.zeros(cout, device=dev),
              running_var=torch.ones(cout, device=dev), num_batches_tracked=torch.zeros((), device=dev, dtype=torch.long),
              mean=torch.empty(cout, device=dev), rstd=torch.empty(cout, device=dev), scale_bias=torch.empty(2 * cout, device=dev),
              eps=1e-5, momentum=0.1)
    for rep in range(2):                        # second launch: self-resetting counters, running statistics advance
        y = C.conv_fprop(x, wt, stride, pad, bn=bn)
    yf = y.float()
    m, v = yf.mean(dim=(0, 2, 3)), yf.var(dim=(0, 2, 3), unbiased=False)
    torch.testing.assert_close(bn["mean"], m, rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(bn["rstd"], torch.rsqrt(v + 1e-5), rtol=1e-3, atol=1e-4)
    sc = bn["gamma"] * torch.rsqrt(v + 1e-5)
    torch.testing.assert_close(bn["scale_bias"][:cout], sc, rtol=1e-3, atol=1e-4)
    torch.testing.assert_close(bn["scale_bias"][cout:], bn["beta"] - m * sc, rtol=1e-3, atol=1e-3)
    cnt = yf.numel() // cout
    torch.testing.assert_close(bn["running_mean"], 0.19 * m, rtol=1e-3, atol=1e-4)
    torch.testing.assert_close(bn["running_var"], 0.81 + 0.19 * v * cnt / (cnt - 1), rtol=1e-3, atol=1e-4)
    assert int(bn["num_batches_tracked"]) == 2


@pytest.mark.parametrize("n,cin,cout,h,w,k,stride,pad", [c for c in CASES if c[6] == 1])
def test_conv_dgrad_matches_fp32(dev, n, cin, cout, h, w, k, stride, pad):
    from vantage6_b200.ops import conv as C

    p, q = h + 2 * pad - k + 1, w + 2 * pad - k + 1
    dy, wt = _t((n, cout, p, q), 5), _t((cout, cin, k, k), 6, (cout * k * k) ** -0.5)
    dx = C.conv_dgrad(dy, wt, (h, w), pad)
    ref = torch.nn.grad.conv2d_input((n, cin, h, w), wt.float(), dy.float(), stride=1, padding=pad)
    torch.testing.assert_close(dx.float(), ref, rtol=2e-2, atol=2e-2)


@pytest.mark.parametrize("n,cin,cout,h,w,k,pad", [(2, 64, 64, 16, 16, 3, 1), (2, 64, 128, 16, 16, 1, 0), (3, 128, 128, 28, 28, 3, 1),
                                                  (3, 256, 512, 28, 28, 1, 0), (5, 512, 512, 14, 14, 3, 1)])
def test_conv_dgrad_stride2_parity_classes(dev, n, cin, cout, h, w, k, pad):
    from vantage6_b200.ops import conv as C

    p, q = (h + 2 * pad - k) // 2 + 1, (w + 2 * pad - k) // 2 + 1
    dy, wt = _t((n, cout, p, q), 15), _t((cout, cin, k, k), 16, (cout * k * k) ** -0.5)
    dx = C.conv_dgrad(dy, wt, (h, w), pad, stride=2)
    ref = torch.nn.grad.conv2d_input((n, cin, h, w), wt.float(), dy.float(), stride=2, padding=pad)
    torch.testing.assert_close(dx.float(), ref, rtol=2e-2, atol=2e-2)


@pytest.mark.parametrize("n,hw", [(2, 32), (4, 224)])
def test_stem_space_to_depth_on_tensor_cores(dev, n, hw):
    """4x4 convolution over the 16-channel space-to-depth image through the overlapping-window im2col map."""
    from vantage6_b200.ops import conv as C

    hs = hw // 2 + 3
    xs, ws = _t((n, 16, hs, hs), 21), _t((64, 16, 4, 4), 22, 1.0 / 16)
    y = C.stem_fprop(xs, ws)
    torch.testing.assert_close(y.float(), F.conv2d(xs.float(), ws.float()), rtol=2e-2, atol=2e-2)
    dy = _t((n, 64, hs - 3, hs - 3), 23, 0.1)
    dws = torch.zeros((64, 4, 4, 16), device=dev)
    C.stem_wgrad(dy, xs, dws)
    ref = torch.nn.grad.conv2d_weight(xs.float(), (64, 16, 4, 4), dy.float()).permute(0, 2, 3, 1)
    torch.testing.assert_close(dws, ref, rtol=1e-3, atol=2e-3 * float(ref.abs().max()))


@pytest.mark.parametrize("n,cin,cout,h,w,k,stride,pad", CASES)
def test_conv_wgrad_accumulates_into_fp32(dev, n, cin, cout, h, w, k, stride, pad):
    from vantage6_b200.ops import conv as C

    p, q = (h + 2 * pad - k) // stride + 1, (w + 2 * pad - k) // stride + 1
    x, dy = _t((n, cin, h, w), 7), _t((n, cout, p, q), 8, 0.1)
    base = torch.randn((cout, k, k, cin), device=dev)
    dw = base.clone()
    C.conv_wgrad(dy, x, dw, (k, k), stride, pad)
    ref = torch.nn.grad.conv2d_weight(x.float(), (cout, cin, k, k), dy.float(), stride=stride, padding=pad).permute(0, 2, 3, 1)
    torch.testing.assert_close(dw - base, ref, rtol=1e-3, atol=2e-3 * float(ref.abs().max()))


@pytest.mark.parametrize("cin,cout,k,splits", [(64, 64, 1, 0), (64, 64, 3, 0), (256, 128, 3, 0), (64, 64, 1, 37)])
def test_split_wgrad_is_the_same_sum_every_run(dev, cin, cout, k, splits):
    """A filter gradient whose K (the pixels) is split over many CTAs: the partial tiles are added in a fixed order, so
    repeated launches give bit-identical results (and still the right ones)."""
    from vantage6_b200.ops import conv as C
    from vantage6_b200.ops import native

    n, hw, pad = 32, 56, k // 2
    assert native().conv_wgrad_workspace(n, hw, hw, cin, cout, k, k, 1, pad, splits) > 0
    x, dy = _t((n, cin, hw, hw), 11), _t((n, cout, hw, hw), 12, 0.1)
    base = torch.randn((cout, k, k, cin), device=dev)
    outs = []
    for _ in range(3):
        dw = base.clone()
        C.conv_wgrad(dy, x, dw, (k, k), 1, pad, splits=splits)
        outs.append(dw)
    assert all(torch.equal(outs[0], o) for o in outs[1:])
    ref = torch.nn.grad.conv2d_weight(x.float(), (cout, cin, k, k), dy.float(), padding=pad).permute(0, 2, 3, 1)
    torch.testing.assert_close(outs[0] - base, ref, rtol=1e-3, atol=2e-3 * float(ref.abs().max()))


def test_resnet_bottleneck_tc_path_matches_cudnn_path(dev, monkeypatch):
    """A ResNet stage through FederatedTrainer-style flat buffers: V6B200_CONV=tc (own kernels, statistics in the
    convolution epilogue, filter gradients straight into the flat buffer) vs V6B200_CONV=cudnn (round-1 path)."""
    from vantage6_b200.models.flat import FlatModel
    from vantage6_b200.models.resnet import Bottleneck
    from vantage6_b200.models.transformer import attach_shadow

    def run(mode):
        monkeypatch.setenv("V6B200_CONV", mode)
        torch.manual_seed(0)
        m = torch.nn.Sequential(Bottleneck(64, 64, 1, _down(64, 256, 1)), Bottleneck(256, 64), Bottleneck(256, 128, 2, _down(256, 512, 2))).to(dev).to(memory_format=torch.channels_last)
        for mod in m.modules():
            if isinstance(mod, Bottleneck):
                torch.nn.init.normal_(mod.bn3.weight, 1.0, 0.1)
        fm = FlatModel(m, shadow=None)
        fm.shadow = fm.flat.to(torch.bfloat16)
        attach_shadow(m, fm)
        m.train()
        x = _t((4, 64, 28, 28), 11).requires_grad_()
        y = m(x)
        (y.float() ** 2).mean().backward()
        fm.flush_grad_sink()
        rm = torch.cat([b.running_mean for b in m.modules() if isinstance(b, torch.nn.BatchNorm2d)])
        return y.detach().float(), x.grad.float(), fm.grad.clone(), rm.clone()

    def _down(cin, cout, stride):
        from vantage6_b200.models.conv import ShadowConv2d
        from vantage6_b200.ops.bn import FusedBatchNormAct

        return torch.nn.Sequential(ShadowConv2d(cin, cout, 1, stride=stride, bias=False), FusedBatchNormAct(cout, relu=False))

    from vantage6_b200.ops import LAUNCHES

    before = LAUNCHES[0]
    y1, dx1, g1, rm1 = run("tc")
    tc_launches = LAUNCHES[0] - before
    y0, dx0, g0, rm0 = run("cudnn")
    assert tc_launches > 0
    # two bf16 pipelines (different summation orders, statistics of the rounded vs unrounded tile): compare in bulk
    diff = (y1 - y0).abs()
    assert float(diff.max()) < 0.25 and float((diff > 5e-2).float().mean()) < 2e-3, (float(diff.max()), float((diff > 5e-2).float().mean()))
    torch.testing.assert_close(rm1, rm0, rtol=1e-2, atol=1e-3)
    assert torch.nn.functional.cosine_similarity(dx1.flatten(), dx0.flatten(), dim=0) > 0.995
    assert torch.nn.functional.cosine_similarity(g1, g0, dim=0) > 0.995
    torch.testing.assert_close(g1.norm(), g0.norm(), rtol=3e-2, atol=1e-4)


def test_side_stream_filter_gradients_match_inline(dev, monkeypatch):
    """Filter gradients issued on the second stream (models/conv.py::_SideWgrad, what the trainer switches on) give the
    gradients of the in-line order; also under CUDA-graph capture, where the fork / join become graph edges."""
    from vantage6_b200.models import conv as CV
    from vantage6_b200.models.flat import FlatModel
    from vantage6_b200.models.resnet import Bottleneck
    from vantage6_b200.models.transformer import attach_shadow

    monkeypatch.setenv("V6B200_CONV", "tc")
    torch.manual_seed(0)
    m = torch.nn.Sequential(Bottleneck(256, 64), Bottleneck(256, 64)).to(dev).to(memory_format=torch.channels_last)
    fm = FlatModel(m, shadow=None)
    fm.shadow = fm.flat.to(torch.bfloat16)
    attach_shadow(m, fm)
    m.train()
    x = _t((8, 256, 28, 28), 5)

    def step(side):
        fm.zero_grad()
        CV.side_wgrad(side)
        try:
            (m(x).float() ** 2).mean().backward()
        finally:
            CV.join_side_wgrad()
            CV.side_wgrad(False)
        fm.flush_grad_sink()

    step(False)
    torch.cuda.synchronize()
    g_inline = fm.grad.clone()
    step(True)
    torch.cuda.synchronize()
    g_side = fm.grad.clone()
    assert float(g_inline.abs().max()) > 0
    torch.testing.assert_close(g_side, g_inline, rtol=1e-3, atol=1e-5 * float(g_inline.abs().max()) + 1e-7)
    # captured: replay twice, the gradients of a replay equal the eager ones
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step(True)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        step(True)
    g.replay()
    g.replay()
    torch.cuda.synchronize()
    torch.testing.assert_close(fm.grad, g_inline, rtol=1e-3, atol=1e-5 * float(g_inline.abs().max()) + 1e-7)
