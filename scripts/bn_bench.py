"""Bandwidth of the BatchNorm passes on the ResNet-50 layer shapes (batch 64).

    PYTHONPATH=. python scripts/bn_bench.py [--out gpurun_out/bn_bench.jsonl]

Prints, per layer shape, the time of every pass (statistics, apply, backward reduce, backward apply), the bytes it has to
move and the resulting GB/s next to the measured copy bandwidth of the box (MEASURED_PEAKS.json).  Buffers rotate over
enough copies to exceed the 126 MB L2.
"""
import argparse
import json

SHAPES = [  # (H=W, C, relu, residual, how many per forward pass)
    (112, 64, True, False, 1),
    (56, 64, True, False, 6), (56, 256, True, True, 3), (56, 256, False, False, 1), (56, 128, True, False, 1),
    (28, 128, True, False, 7), (28, 512, True, True, 4), (28, 512, False, False, 1), (28, 256, True, False, 1),
    (14, 256, True, False, 11), (14, 1024, True, True, 6), (14, 1024, False, False, 1), (14, 512, True, False, 1),
    (7, 512, True, False, 5), (7, 2048, True, True, 3), (7, 2048, False, False, 1),
]


def bench():
    import torch

    from vantage6_b200.ops import native, stream_ptr
    from vantage6_b200.ops.bn import _get_scratch

    C_ = native()
    dev = torch.device("cuda", 0)
    N = 64

    def timeit(fn, nset, iters=24):
        for i in range(4):
            fn(i % nset)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(iters):
            fn(i % nset)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters * 1e3        # us

    tot = {"stats": 0.0, "apply": 0.0, "bwd_reduce+apply": 0.0}
    lines = []
    for (hw, C, relu, res, mult) in SHAPES:
        R = N * hw * hw
        nbytes = R * C * 2
        nset = max(2, min(8, int(400e6 // (nbytes * 4)) + 1))
        mk = lambda: [torch.randn(R, C, device=dev).to(torch.bfloat16) for _ in range(nset)]   # noqa: E731
        x, dy, y, dx = mk(), mk(), mk(), mk()
        rs = mk() if res else None
        dres = mk() if res else None
        mask = [torch.empty(R, C // 8, device=dev, dtype=torch.uint8) for _ in range(nset)]
        gamma, beta = torch.rand(C, device=dev) + 0.5, torch.randn(C, device=dev)
        mean, rstd, sb = torch.empty(C, device=dev), torch.empty(C, device=dev), torch.empty(2 * C, device=dev)
        dg, db = torch.zeros(C, device=dev), torch.zeros(C, device=dev)
        part, coef = _get_scratch(dev, C)
        s = stream_ptr()

        def fwd(i):
            C_.bn_fwd(x[i].data_ptr(), rs[i].data_ptr() if res else 0, gamma.data_ptr(), beta.data_ptr(), 0, 0, 0, y[i].data_ptr(),
                      mask[i].data_ptr() if relu else 0, mean.data_ptr(), rstd.data_ptr(), sb.data_ptr(), part.data_ptr(), R, C, 1e-5, 0.1, relu, s)

        def apply(i):
            C_.bn_apply(x[i].data_ptr(), rs[i].data_ptr() if res else 0, sb.data_ptr(), sb.data_ptr() + 4 * C, y[i].data_ptr(),
                        mask[i].data_ptr() if relu else 0, R, C, relu, s)

        def bwd(i):
            C_.bn_bwd(dy[i].data_ptr(), mask[i].data_ptr() if relu else 0, x[i].data_ptr(), gamma.data_ptr(), mean.data_ptr(), rstd.data_ptr(),
                      dx[i].data_ptr(), dres[i].data_ptr() if res else 0, dg.data_ptr(), db.data_ptr(), coef.data_ptr(), part.data_ptr(), R, C,
                      relu, False, s)

        t_fwd, t_apply, t_bwd = timeit(fwd, nset), timeit(apply, nset), timeit(bwd, nset)
        mb = nbytes / 8 if relu else 0
        b_apply = nbytes * (2 + (1 if res else 0)) + mb
        b_bwd = (2 * nbytes + mb) * 2 + nbytes * (1 + (1 if res else 0))
        rec = dict(hw=hw, C=C, relu=relu, res=res, mult=mult, mb_per_tensor=nbytes / 1e6, stats_us=t_fwd - t_apply, apply_us=t_apply,
                   apply_gbs=b_apply / t_apply * 1e-3, stats_gbs=nbytes / max(t_fwd - t_apply, 1e-3) * 1e-3, bwd_us=t_bwd, bwd_gbs=b_bwd / t_bwd * 1e-3)
        print(json.dumps(rec), flush=True)
        lines.append(json.dumps(rec))
        tot["stats"] += mult * (t_fwd - t_apply)
        tot["apply"] += mult * t_apply
        tot["bwd_reduce+apply"] += mult * t_bwd
        del x, dy, y, dx, rs, dres, mask
    lines.append(json.dumps(dict(per_step_ms={k: v / 1e3 for k, v in tot.items()})))
    print(lines[-1], flush=True)
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    lines = bench()
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
