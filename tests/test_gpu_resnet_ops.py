"""ResNet-50 local-step pieces on the GPU: max-pool / image-normalise kernels, the multi-tensor gradient sink,
ShadowConv2d (bf16 shadow filters + gradient sink) against the autocast path, in-kernel BN reduction trees."""
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    from vantage6_b200.ops import native

    native()
    torch.cuda.set_device(0)
    return torch.device("cuda", 0)


@pytest.mark.parametrize("N,C,H,W", [(4, 64, 112, 112), (2, 8, 9, 7), (3, 16, 32, 32), (1, 64, 5, 5)])
def test_maxpool_matches_torch(dev, N, C, H, W):
    from vantage6_b200.ops.pool import MaxPool3x3s2

    torch.manual_seed(0)
    x = torch.randn(N, C, H, W, device=dev).to(torch.bfloat16).contiguous(memory_format=torch.channels_last).requires_grad_()
    y = MaxPool3x3s2()(x)
    dy = torch.randn_like(y)
    y.backward(dy)
    xr = x.detach().float().requires_grad_()
    yr = torch.nn.functional.max_pool2d(xr, 3, 2, 1)
    yr.backward(dy.float())
    assert y.shape == yr.shape and y.is_contiguous(memory_format=torch.channels_last)
    torch.testing.assert_close(y.float(), yr, rtol=0, atol=0)
    # ties (equal bf16 values inside a window) may pick a different arg-max than the fp32 reference only when
    # values are exactly equal; the routed gradient mass is identical either way
    torch.testing.assert_close(x.grad.float().sum(), xr.grad.sum(), rtol=1e-2, atol=1e-1)
    mism = (x.grad.float() - xr.grad).abs() > 2e-2
    assert mism.float().mean().item() < 2e-3


def test_image_normalize_matches_torch(dev):
    from vantage6_b200.models.resnet import _MEAN, _STD
    from vantage6_b200.ops.pool import image_normalize

    g = torch.Generator().manual_seed(1)
    img = torch.randint(0, 256, (5, 3, 64, 48), dtype=torch.uint8, generator=g).to(dev)
    out = image_normalize(img, _MEAN, _STD)
    m = torch.tensor(_MEAN, device=dev).view(1, 3, 1, 1)
    s = torch.tensor(_STD, device=dev).view(1, 3, 1, 1)
    ref = ((img.float() - m) / s).to(torch.bfloat16)
    assert out.shape == img.shape and out.is_contiguous(memory_format=torch.channels_last)
    torch.testing.assert_close(out.float(), ref.float(), rtol=1e-2, atol=1e-2)


def test_multi_accumulate(dev):
    from vantage6_b200.ops.optim import multi_accumulate

    torch.manual_seed(2)
    sizes = [8, 4096, 9408, 64 * 64 * 9, 2048 * 512, 24] + [128] * 120       # > 96 tensors: two launches
    offs, o = [], 0
    for n in sizes:
        offs.append(o)
        o += (n + 7) // 8 * 8
    dst = torch.randn(o, device=dev)
    ref = dst.clone()
    items = []
    for n, off in zip(sizes, offs):
        g = torch.randn(n, device=dev).to(torch.bfloat16)
        items.append((g, off))
        ref[off: off + n] += g.float()
    multi_accumulate(dst, items)
    torch.testing.assert_close(dst, ref, rtol=0, atol=0)


def test_bn_large_shapes_repeatable(dev):
    """Two-level reduction trees (many row-CTAs per slice); counters must reset: run twice, bitwise equal."""
    from vantage6_b200.ops.bn import FusedBatchNormAct

    for (N, C, H, W) in [(64, 64, 56, 56), (32, 256, 56, 56), (64, 2048, 7, 7), (64, 512, 28, 28)]:
        torch.manual_seed(3)
        x = (torch.randn(N, C, H, W, device=dev) * 1.5 - 0.3).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
        bn = FusedBatchNormAct(C).to(dev)
        outs = []
        for _ in range(3):
            xi = x.clone().requires_grad_()
            y = bn(xi)
            y.backward(torch.ones_like(y))
            outs.append((y.detach().clone(), xi.grad.clone(), bn.weight.grad.clone()))
            bn.weight.grad = None
            bn.bias.grad = None
        for a, b in zip(outs[0], outs[2]):
            assert torch.equal(a, b)
        xf = x.float()
        mean = xf.mean((0, 2, 3))
        var = xf.var((0, 2, 3), unbiased=False)
        ref = torch.relu((xf - mean.view(1, -1, 1, 1)) * torch.rsqrt(var + bn.eps).view(1, -1, 1, 1))
        torch.testing.assert_close(outs[0][0].float(), ref, rtol=2e-2, atol=2e-2)
        assert int(bn.num_batches_tracked) == 3


def test_resnet_shadow_conv_trainer_matches_autocast(dev):
    """Same seeds, fused arm (ShadowConv2d + gradient sink + fused BN/pool + K7 + CUDA graph) vs the stock arm."""
    from vantage6_b200.models import zoo

    def run(fused):
        torch.manual_seed(11)
        tr, spec = zoo.build_trainer("resnet_tiny", rank=0, world=1, device=dev, data_plane="auto" if fused else "collective",
                                     fused_local_optimizer=fused, use_cuda_graph=fused)
        batches = spec.make_batches(2, 8, 1234, pin=True)
        tr.initialize_global()
        losses = [float(tr.run_round(batches, 16.0).item()) for _ in range(4)]
        shadow_ok = True
        if fused:
            nt = tr.fm.n_trainable
            shadow_ok = torch.equal(tr.engine.shadow[:nt], tr.engine.w[:nt].to(torch.bfloat16))
            from vantage6_b200.models.conv import ShadowConv2d

            assert all(m.w_bf16 is not None for m in tr.model.modules() if isinstance(m, ShadowConv2d))
        tr.close()
        return losses, shadow_ok

    a, ok = run(True)
    b, _ = run(False)
    assert ok
    assert abs(a[0] - b[0]) < 0.08 and abs(a[-1] - b[-1]) < 0.35, (a, b)


@pytest.mark.parametrize("N,H,W,O", [(2, 64, 64, 8), (3, 224, 224, 64), (1, 32, 48, 16)])
def test_stem_space_to_depth_matches_direct_conv(dev, N, H, W, O):
    """4x4/s1 conv on the space-to-depth image == 7x7/s2/p3 conv on the normalised image (values and filter grads)."""
    from vantage6_b200.models.resnet import _MEAN, _STD
    from vantage6_b200.ops import pool

    g = torch.Generator().manual_seed(4)
    img = torch.randint(0, 256, (N, 3, H, W), dtype=torch.uint8, generator=g).to(dev)
    conv = torch.nn.Conv2d(3, O, 7, stride=2, padding=3, bias=False).to(dev).to(memory_format=torch.channels_last)
    assert pool.stem_s2d_supported(img, conv)
    y = pool.stem_s2d(img, conv, _MEAN, _STD)
    dy = torch.randn_like(y)
    y.backward(dy)
    got_dw = conv.weight.grad.clone()
    conv.weight.grad = None
    m = torch.tensor(_MEAN, device=dev).view(1, 3, 1, 1)
    s = torch.tensor(_STD, device=dev).view(1, 3, 1, 1)
    xn = ((img.float() - m) / s).to(torch.bfloat16).float()
    wr = conv.weight.detach().to(torch.bfloat16).float().requires_grad_()
    yr = torch.nn.functional.conv2d(xn, wr, None, 2, 3)
    yr.backward(dy.float())
    assert y.shape == yr.shape and y.is_contiguous(memory_format=torch.channels_last)
    torch.testing.assert_close(y.float(), yr, rtol=2e-2, atol=2e-2)
    scale = wr.grad.abs().max().item()
    assert (got_dw - wr.grad).abs().max().item() < 2e-2 * scale
    # accumulate-into-existing-grad path
    conv.weight.grad = torch.ones_like(conv.weight, memory_format=torch.channels_last)
    y2 = pool.stem_s2d(img, conv, _MEAN, _STD)
    y2.backward(dy)
    assert ((conv.weight.grad - 1.0) - wr.grad).abs().max().item() < 2e-2 * scale


@pytest.mark.parametrize("N,C,H,W", [(4, 64, 112, 112), (2, 64, 10, 14), (3, 128, 16, 16)])
def test_stem_bn_apply_maxpool_matches_torch(dev, N, C, H, W):
    """Stem tail: BatchNorm apply + ReLU with the statistics of the producing convolution (``apply_pre``), then the 3x3 / s2
    max-pool, against ``max_pool2d(relu(x * scale + bias))`` in fp32 PyTorch: the output, dx, dgamma and dbeta."""
    from vantage6_b200.ops import bn as BN
    from vantage6_b200.ops.pool import MaxPool3x3s2

    torch.manual_seed(0)
    x0 = torch.randn(N, C, H, W, device=dev).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    bnm = BN.FusedBatchNormAct(C, relu=True).to(dev)
    with torch.no_grad():
        bnm.weight.uniform_(0.5, 1.5)
        bnm.bias.normal_(0, 0.3)
    bnm.train()

    def affine(x, gamma, beta):
        mean = x.mean((0, 2, 3))
        rstd = torch.rsqrt(x.var((0, 2, 3), unbiased=False) + bnm.eps)
        return mean, rstd, gamma * rstd, beta - mean * gamma * rstd

    mean, rstd, scale, bias = affine(x0.float(), bnm.weight.detach(), bnm.bias.detach())
    stats = dict(mean=mean.contiguous(), rstd=rstd.contiguous(), scale_bias=torch.cat([scale, bias]).contiguous(), momentum=0.1)

    xa = x0.clone().requires_grad_()
    y = MaxPool3x3s2()(bnm.apply_pre(xa, stats))
    dy = torch.randn_like(y)
    y.backward(dy)
    torch.cuda.synchronize()

    # the kernel rounds fmaf(x, scale, bias) to bf16.  In fp64 the product of a bf16 and an fp32 value is exact and the sum keeps
    # 29 bits more than fp32, so t rounds to the same fp32 value, and its sign is the ReLU decision the kernel made
    with torch.no_grad():
        t = x0.double() * scale.double().view(1, -1, 1, 1) + bias.double().view(1, -1, 1, 1)
        y1 = torch.relu(t).float().to(torch.bfloat16).float()
        keep = (t > 0).float()
    torch.testing.assert_close(y.float(), torch.nn.functional.max_pool2d(y1, 3, 2, 1), rtol=0, atol=0)

    # backward: BatchNorm with batch statistics (mean and variance are functions of x) in fp32; the pooled values are the
    # kernel's bf16 ones (straight-through), so that max_pool2d picks the same window maxima and routes dy to the same pixels
    xr = x0.float().requires_grad_()
    gr = bnm.weight.detach().clone().requires_grad_()
    br = bnm.bias.detach().clone().requires_grad_()
    _, _, sr, bir = affine(xr, gr, br)
    lin = (xr * sr.view(1, -1, 1, 1) + bir.view(1, -1, 1, 1)) * keep
    lin = lin + (y1 - lin).detach()
    torch.nn.functional.max_pool2d(lin, 3, 2, 1).backward(dy.float())
    torch.testing.assert_close(bnm.weight.grad, gr.grad, rtol=2e-3, atol=2e-3 * float(gr.grad.abs().max()))
    torch.testing.assert_close(bnm.bias.grad, br.grad, rtol=2e-3, atol=2e-3 * float(br.grad.abs().max()))
    d = (xa.grad.float() - xr.grad).abs()
    assert float(d.max()) <= 2e-2 * float(xr.grad.abs().max()) + 1e-6, float(d.max())
