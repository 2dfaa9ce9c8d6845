#!/usr/bin/env python
"""Headline benchmark (BASELINE.json): federated rounds/sec for ResNet-50 FedAvg, one federated
node per GPU, 1 local epoch per round on synthetic ImageNet-shape data, random-init weights -- and, with
``--model``, the other BASELINE.json configs (BERT-base bf16 4 local steps/round, Llama-3 8B LoRA, logistic GLM).

    python bench.py --gpus N --steps K --warmup W            # product arm, then the same-box comparator arms
    python bench.py --impl nccl ...                          # only the in-repo NCCL + cuDNN/cuBLAS + torch.optim arm
    python bench.py --impl stock_graph ...                   # stock layers / torch.optim / NCCL, local step in ONE CUDA graph
    python bench.py --impl reference ...                     # the unmodified reference (unavailable, see DESIGN.md)
    python bench.py --model bert_base|llama3_8b_lora|glm ...
    python bench.py --dump-outputs DIR ...                   # also write the last timed step's outputs as DIR/<name>.npy

A bench "step" is ONE federated round = `local_steps` local optimizer steps on every node + the server aggregation
(weighted FedAvg reduce + server optimizer + broadcast of the new global); for the GLM one step is one federated
gradient iteration.  `value` = nodes x rounds/sec (the whole-job aggregate: node-local epochs completed per second
across the federation; `rounds_per_sec` is printed next to it).  Weak scaling: per-node work is fixed.

The reference cannot run here (it is a Docker-launching CLI with no compute, DESIGN.md section 4), so the line of the
product arm carries the same-box comparison itself: after the product arm the SAME process group runs the comparator
arms with the same steps / warm-up / data / init and `vs_baseline` = product value / NCCL-arm value
(details of every arm under `baseline_arms`).

Timing: W untimed warm-up rounds, then exactly K rounds between CUDA events, bracketed by barrier +
torch.cuda.synchronize() on both sides, max over ranks.  Inputs per round exceed the 126 MB L2 (ResNet-50: 77 MB of
images + 102 MB of model + GBs of activations), so no flush is needed between rounds.  `e2e` repeats the measurement
through the public API (`FederatedTrainer.run_round`) with the round's batches living in pinned host memory (H2D copy
every local step) and a device->host read of the round's loss.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODELS = ["resnet50", "resnet_tiny", "resnet_mini", "bert_base", "bert_tiny", "llama3_8b_lora", "llama_tiny_lora", "glm"]


def parse(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8, help="timed federated rounds")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "nccl", "stock_graph", "reference"])
    ap.add_argument("--model", default="resnet50", choices=MODELS)
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--local-samples", type=int, default=512, help="ResNet: node-local dataset size = 1 epoch")
    ap.add_argument("--local-steps", type=int, default=None)
    ap.add_argument("--server-mode", default="sharded", choices=["sharded", "central"])
    ap.add_argument("--server-opt", default="fedavg", choices=["fedavg", "fedavgm", "fedadam"])
    ap.add_argument("--baselines", default=None, help="comma list of comparator arms run after the product arm "
                                                      "(default: nccl,stock_graph for ResNet, nccl otherwise; '' = none)")
    ap.add_argument("--bcast", default=os.environ.get("V6B200_BCAST", "push"), choices=["push", "fused"],
                    help="fused: K1 -- the first-consumer weights arrive inside the first forward GEMM of the round (transformers, >= 2 GPUs)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the measured arm computed in its last step (the round's loss and "
                         "the new global model; for the GLM the loss and coefficients) as float32 DIR/<name>.npy")
    return ap.parse_args(argv)


DUMP_MAX_ELEMS = 1 << 23        # 32 MB of float32: a larger output is written as a fixed, seeded sample of its elements


def dump_outputs(out_dir, arrays):
    """Write each tensor of ``arrays`` as float32 ``out_dir/<name>.npy``.  The sample of an output larger than
    DUMP_MAX_ELEMS takes the same (sorted) flat indices on every run, so two builds can be compared element for element."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_MAX_ELEMS:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ELEMS].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(out_dir, f"{name}.npy"), t.float().cpu().numpy())


def reference_unavailable():
    if int(os.environ.get("RANK", "0")) == 0:           # one line, from rank 0 only (N > 1 runs under torchrun)
        print(json.dumps({
            "impl": "reference",
            "unavailable": "reference snapshot is only the vantage6 CLI: --no-deps install imports fail "
                           "(questionary, docker, schema, vantage6.common, vantage6.client missing offline); it has no "
                           "FedAvg/NCCL/GPU path to time and needs a Docker daemon (see DESIGN.md)"}), flush=True)


# ------------------------------------------------------------------------------------------------- arms
def build_trainer(impl, args, rank, world, device):
    """-> (trainer, batches factory info).  impl: b200 | nccl | stock_graph."""
    import torch

    from vantage6_b200.parallel.fedavg import ServerOptConfig

    b200 = impl == "b200"
    graph = (b200 and not args.no_graph) or impl == "stock_graph"
    sopt = ServerOptConfig(args.server_opt, 1.0)
    if args.model.startswith("resnet"):
        from vantage6_b200.models import resnet as R
        from vantage6_b200.parallel.trainer import FederatedTrainer

        # product arm: hand-written conv / fused BN(+add)(+ReLU) kernels; comparator arms: stock Conv2d/BatchNorm2d/ReLU/add
        if args.model == "resnet50":
            model = R.resnet50(fused_bn=b200)
        elif args.model == "resnet_mini":
            model = R.ResNet((1, 1, 1, 1), 1000, fused_bn=b200)
        else:
            model = R.resnet_tiny(1000, fused_bn=b200)
        model = model.to(memory_format=torch.channels_last)
        tr = FederatedTrainer(
            model, R.imagenet_forward_loss, rank=rank, world=world, device=device, optimizer="sgd", lr=0.05, momentum=0.9,
            weight_decay=1e-4, server_mode=args.server_mode, server_opt=sopt, upload="weights_f32",
            data_plane="native" if b200 else "collective", use_cuda_graph=graph, fused_local_optimizer=b200,
            amp_dtype=torch.bfloat16, shadow_bf16=b200)     # product arm: filters are consumed from the bf16 shadow kept by K7 / K2
        return tr, None
    from vantage6_b200.models import zoo

    tr, spec = zoo.build_trainer(args.model, rank=rank, world=world, device=device, server_mode=args.server_mode,
                                 server_opt=sopt, data_plane="native" if b200 else "collective", fused_local_optimizer=b200,
                                 use_cuda_graph=graph, **({"bcast": "fused"} if (b200 and args.bcast == "fused") else {}))
    return tr, spec


def make_data(args, spec, rank, device):
    """Pinned host batches + device copies of one node's (non-IID, synthetic) local epoch."""
    import torch

    if spec is None:
        B = args.batch or 64
        n_steps = args.local_steps or max(1, args.local_samples // B)
        res = {"resnet50": 224, "resnet_mini": 64}.get(args.model, 64)
        g = torch.Generator().manual_seed(100 + rank)
        host_x = torch.randint(0, 256, (n_steps, B, 3, res, res), dtype=torch.uint8, generator=g).pin_memory()
        host_y = torch.randint(0, 1000, (n_steps, B), dtype=torch.int64, generator=g).pin_memory()
        host = [(host_x[i], host_y[i]) for i in range(n_steps)]
        shape = {"image": [3, res, res], "seq_len": None}
    else:
        B = args.batch or spec.batch
        n_steps = args.local_steps or spec.local_steps
        host = spec.make_batches(n_steps, B, seed=500 + rank, pin=True)
        shape = {"seq_len": int(host[0][0].shape[1]) if host[0][0].dim() == 2 else None}
    dev = [(x.to(device), y.to(device)) for x, y in host]
    h2d = sum(x.numel() * x.element_size() + y.numel() * y.element_size() for x, y in host)
    return host, dev, B, n_steps, h2d, shape


def run_trainer_arm(impl, args, rank, world, local_rank, device):
    import torch

    from vantage6_b200.utils.timing import ClockSampler, DeviceTimer, barrier_sync, max_over_ranks

    torch.manual_seed(1234)           # identical random init everywhere (rank 0's is authoritative)
    trainer, spec = build_trainer(impl, args, rank, world, device)
    trainer.initialize_global()
    host, dev, B, n_steps, h2d, shape = make_data(args, spec, rank, device)
    n_samples = float(n_steps * B)

    def run(batches, rounds, read_loss):
        last = None
        for _ in range(rounds):
            last = trainer.run_round(batches, n_samples)
            if read_loss:
                last = last.item()          # device -> host read of the round's result
        return last

    run(dev, args.warmup, False)
    barrier_sync(device)
    timer = DeviceTimer(device)
    with ClockSampler(local_rank) as clocks:
        barrier_sync(device)
        launches0 = trainer.native_launches
        timer.start()
        torch.cuda.nvtx.range_push("v6_timed")          # ncu --nvtx --nvtx-include "v6_timed/"
        loss = run(dev, args.steps, False)
        launches = trainer.native_launches - launches0
        torch.cuda.nvtx.range_pop()
        ms = timer.stop()
        barrier_sync(device)
    ms = max_over_ranks(ms, device)
    if args.dump_outputs and impl == args.impl and rank == 0:       # before the aggregation-only and e2e passes move the model
        dump_outputs(args.dump_outputs, {"loss": loss, "global_model": trainer.fm.flat[: trainer.fm.n_total]})
    loss_val = float(loss.item())
    if os.environ.get("V6_PROFILE_RANGE") and impl == "b200":      # ncu --profile-from-start off: one more round
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        run(dev, 1, False)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
    status = trainer.engine.poll_status()
    # aggregation alone (the communication-bound part of the round)
    eng = trainer.engine
    snap = [t.clone() for t in (eng.w, eng.w_global, eng.opt_m, eng.opt_v)] + [eng.server_step]
    barrier_sync(device)
    timer.start()
    for _ in range(10):
        eng.aggregate(1.0)
    agg_ms = max_over_ranks(timer.stop(), device) / 10
    for dst, src in zip((eng.w, eng.w_global, eng.opt_m, eng.opt_v), snap[:4]):
        dst.copy_(src)                      # the extra aggregations must not leak into the end-to-end measurement
    eng.server_step = snap[4]
    if eng.shadow is not None:
        eng.shadow.copy_(eng.w.to(torch.bfloat16))

    e2e = None
    if not args.no_e2e:
        run(host, 1, True)
        barrier_sync(device)
        t0 = time.perf_counter()
        run(host, args.steps, True)
        barrier_sync(device)
        e2e_s = max_over_ranks(time.perf_counter() - t0, device)
        e2e = {"value": world * args.steps / e2e_s, "unit": "node-rounds/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": 4, "ms_per_step": 1e3 * e2e_s / args.steps}
    rps = args.steps / (ms / 1e3)
    nv = trainer.engine.nvlink_bytes_per_round()
    out = {"impl": impl, "value": world * rps, "ms_per_step": ms / args.steps, "rounds_per_sec": rps,
           "samples_per_sec": world * rps * n_samples, "e2e": e2e, "gpu_launches": int(launches), "final_loss": loss_val,
           "comm_status": status, "aggregate_ms": agg_ms, "nvlink_bytes_per_round_per_gpu": nv,
           "aggregate_bus_GBps": (nv / (agg_ms * 1e-3) / 1e9) if (nv and agg_ms) else None,
           "clocks": clocks.summary(),
           "config": {"model": args.model, "global_batch": B * world, "parallelism": f"fedavg{world} (1 node/GPU, server {args.server_mode})",
                      "local_steps_per_round": n_steps, "local_batch": B, "local_samples": int(n_samples), **shape,
                      "server_opt": args.server_opt, "param_dtype": "fp32 master", "upload": trainer.upload_mode,
                      "bcast": ("fused (K1: %d layers)" % trainer.k1_layers) if getattr(trainer, "k1_layers", 0) else "push (K2)",
                      "n_federated_params": int(trainer.fm.n_total),
                      "l2": "inputs larger than L2 (per-round inputs + model + activations >> 126 MB), no flush",
                      "data_plane": trainer.engine.data_plane, "multicast": bool(trainer.engine.use_multicast),
                      "cuda_graph": bool(trainer.use_graph), "conv": os.environ.get("V6B200_CONV", "tc") if impl == "b200" else "cudnn"}}
    trainer.close()
    return out


def run_glm_arm(impl, args, rank, world, local_rank, device):
    """BASELINE config 5: logistic GLM on 1M x 256 synthetic rows split over the nodes; one step = one federated gradient
    iteration (local gradient + loss over the shard -> small-message aggregation -> coefficient update)."""
    import torch
    import torch.distributed as dist

    from vantage6_b200.models.glm import FederatedGLM, synthetic_glm_shard
    from vantage6_b200.ops import LAUNCHES
    from vantage6_b200.utils.timing import ClockSampler, DeviceTimer, barrier_sync, max_over_ranks

    rows = 1_000_000 // max(world, 1)
    X, y, w_true = synthetic_glm_shard(rows, 256, seed=100 + rank, device=device)
    if impl == "b200":
        glm = FederatedGLM(X, y, rank, world, lr=2.0)
        step, coef = glm.step, glm.w
    else:       # comparator: two cuBLAS GEMVs + elementwise + ncclAllReduce of the 259-float payload
        w = coef = torch.zeros(257, device=device)

        def step():
            z = (X @ w[:256].to(X.dtype)).float() + w[256]
            r = torch.sigmoid(z) - y
            g = torch.cat([(X.t() @ r.to(X.dtype)).float(), r.sum()[None],
                           torch.nn.functional.binary_cross_entropy_with_logits(z, y, reduction="sum")[None],
                           torch.tensor([float(rows)], device=device)])
            if world > 1:
                dist.all_reduce(g)
            w.add_(g[:257] / g[258], alpha=-2.0)
            return g[257] / g[258]
    for _ in range(max(args.warmup, 3) * 5):
        step()
    iters = args.steps * 25                        # a "step" of the GLM bench = 25 iterations (each ~0.1 ms)
    barrier_sync(device)
    t = DeviceTimer(device)
    with ClockSampler(local_rank) as clocks:
        barrier_sync(device)
        l0 = LAUNCHES[0]
        t.start()
        for _ in range(iters):
            loss = step()
        ms = max_over_ranks(t.stop(), device)
        launches = LAUNCHES[0] - l0
    if args.dump_outputs and impl == args.impl and rank == 0:
        dump_outputs(args.dump_outputs, {"loss": loss, "coefficients": coef})
    t0 = time.perf_counter()
    for _ in range(iters):
        lv = float(step().item())                  # end to end: the iteration's loss is read back every iteration
    e2e_s = max_over_ranks(time.perf_counter() - t0, device)
    ips = iters / (ms / 1e3)
    return {"impl": impl, "value": world * ips, "ms_per_step": ms / iters, "rounds_per_sec": ips, "us_per_iteration": 1e3 * ms / iters,
            "samples_per_sec": world * ips * rows, "X_read_GBps": rows * 256 * 2 / (ms / iters) / 1e6,
            "e2e": {"value": world * iters / e2e_s, "unit": "node-iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 4,
                    "ms_per_step": 1e3 * e2e_s / iters, "note": "the node's shard is resident (full-batch GD re-reads it every iteration)"},
            "gpu_launches": int(launches), "final_loss": lv, "comm_status": 0, "clocks": clocks.summary(),
            "config": {"model": "glm", "global_batch": rows * world, "seq_len": None, "rows_per_node": rows, "features": 256,
                       "parallelism": f"fedavg{world} (1 node/GPU, small-message aggregation)", "iterations_timed": iters,
                       "l2": "the 512 MB shard exceeds L2, no flush"}}


def main():
    args = parse()
    if args.impl == "reference":
        reference_unavailable()
        return 0

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and rank == 0:
        print(f"[bench] note: WORLD_SIZE={world} overrides --gpus {args.gpus}", file=sys.stderr)
    if not torch.cuda.is_available():
        print(json.dumps({"metric": "federated_node_rounds_per_sec", "value": None, "unit": "node-rounds/s",
                          "error": "no CUDA device visible"}))
        return 1
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    torch.backends.cudnn.benchmark = True
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.allow_tf32 = True

    arm = run_glm_arm if args.model == "glm" else run_trainer_arm
    main_res = arm(args.impl, args, rank, world, local_rank, device)
    arms = {}
    if args.impl == "b200":
        default = "nccl,stock_graph" if args.model.startswith("resnet") else "nccl"
        wanted = [a for a in (default if args.baselines is None else args.baselines).split(",") if a]
        if args.model == "glm":
            wanted = [a for a in wanted if a == "nccl"]
        for a in wanted:
            try:
                arms[a] = arm(a, args, rank, world, local_rank, device)
            except Exception as e:  # noqa: BLE001 -- a failing comparator must not take the product line down
                arms[a] = {"impl": a, "error": repr(e)[:300]}
    if rank == 0:
        unit = "node-iterations/s" if args.model == "glm" else "node-rounds/s"
        name = {"resnet50": "ResNet-50", "bert_base": "BERT-base", "llama3_8b_lora": "Llama-3 8B LoRA", "glm": "logistic GLM 1Mx256"}.get(args.model, args.model)
        base = arms.get("nccl") if "value" in arms.get("nccl", {}) else None
        out = {
            "metric": f"federated_node_rounds_per_sec ({name} FedAvg, rounds/sec x nodes)",
            "value": main_res["value"], "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": main_res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": (main_res["value"] / base["value"]) if base else None,
            "vs_baseline_note": (("value / same-box comparator arm run in this process after the product arm: " + (
                "stock torchvision-style model (cuDNN convolutions, stock BatchNorm / ReLU / pooling), torch.optim, NCCL aggregation"
                if args.model.startswith("resnet") else
                "two cuBLAS GEMVs + elementwise ops + ncclAllReduce per iteration" if args.model == "glm" else
                "the same model code WITHOUT the bf16 shadow (per-step casts), torch.optim, NCCL reduce + broadcast -- its forward still runs "
                "on this repo's GEMM / attention / norm kernels, so the ratio understates the distance to a stock PyTorch model")
                + " (BASELINE.md: the reference publishes no number and cannot run)") if base else None),
            "dtype": "bf16", "data": "synthetic", "impl": args.impl,
            "rounds_per_sec": main_res["rounds_per_sec"], "node_rounds_per_sec": main_res["value"],
            "samples_per_sec": main_res.get("samples_per_sec"),
            "config": main_res["config"], "clocks": main_res["clocks"], "e2e": main_res["e2e"],
            "gpu_launches": main_res["gpu_launches"], "final_loss": main_res["final_loss"], "comm_status": main_res["comm_status"],
        }
        for k in ("aggregate_ms", "nvlink_bytes_per_round_per_gpu", "aggregate_bus_GBps", "us_per_iteration", "X_read_GBps"):
            if k in main_res:
                out[k] = main_res[k]
        if base and main_res.get("e2e") and base.get("e2e"):
            out["vs_baseline_e2e"] = main_res["e2e"]["value"] / base["e2e"]["value"]
        if arms:
            out["baseline_arms"] = {
                a: ({k: r.get(k) for k in ("value", "ms_per_step", "rounds_per_sec", "e2e", "final_loss", "aggregate_ms", "clocks", "error")
                     if r.get(k) is not None} | ({"ratio": main_res["value"] / r["value"]} if r.get("value") else {}))
                for a, r in arms.items()}
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
