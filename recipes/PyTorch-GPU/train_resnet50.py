#!/usr/bin/env python3
"""PyTorch-GPU recipe body (north-star retarget): multi-instance ResNet-50 training, one rank per GPU.

The reference recipe launches a stock PyTorch MNIST container on one K80
(/root/reference/recipes/PyTorch-GPU/config/jobs.yaml:1-8).  Here the task runner starts one
rank per GPU (RANK / WORLD_SIZE / SHIPYARD_GPU in the environment) and the step runs on the
fused trainer: flat symmetric parameters, one fused all-reduce+SGD+all-gather kernel per step,
CUDA-graph captured, uint8 batches staged from pinned memory.
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.environ.get("SHIPYARD_HOME") or os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))

import torch  # noqa: E402

from batch_shipyard_b200.models.resnet import resnet50, resnet_tiny  # noqa: E402
from batch_shipyard_b200.ops.coll import Communicator  # noqa: E402
from batch_shipyard_b200.parallel.ddp import FusedDataParallelTrainer  # noqa: E402


def _held_out(a, rank, nclass):
    """a.eval_batches x a.batch held-out uint8 NHWC images and labels for this rank (seeded, disjoint from the training seeds)."""
    n = a.eval_batches * a.batch
    seed = 555000 + rank
    if a.model == "lenet":
        from batch_shipyard_b200.models.lenet import synthetic_digits
        return synthetic_digits(n, seed=seed)
    if a.model == "resnet20":
        from batch_shipyard_b200.models.resnet import synthetic_cifar
        return synthetic_cifar(n, seed=seed)
    g = torch.Generator().manual_seed(seed)
    return (torch.randint(0, 256, (n, a.image, a.image, 3), dtype=torch.uint8, generator=g),
            torch.randint(0, nclass, (n,), dtype=torch.int64, generator=g))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--batch", type=int, default=256, help="per-GPU batch")
    ap.add_argument("--image", type=int, default=224)
    ap.add_argument("--model", default="resnet50", choices=["resnet50", "tiny", "lenet", "resnet20"],
                    help="resnet50 (the GPU recipes), tiny (a 4-block ResNet for smoke runs), lenet (the MNIST network of the single-framework CPU recipes, synthetic digits), resnet20 (the CIFAR-10 ResNet of the MXNet / CNTK examples, synthetic CIFAR-shaped images)")
    ap.add_argument("--lr", type=float, default=0.1)
    ap.add_argument("--eval-batches", type=int, default=0,
                    help="after training, evaluate on this many held-out seeded batches per rank (FusedDataParallelTrainer.evaluate; "
                         "the sums of all ranks are reported under \"eval\")")
    a = ap.parse_args()
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    gpu = os.environ.get("SHIPYARD_GPU", os.environ.get("LOCAL_RANK", "0"))
    use_cuda = torch.cuda.is_available() and gpu not in ("", "-1")
    dev_index = int(gpu) % max(1, torch.cuda.device_count()) if use_cuda else None
    if use_cuda:
        torch.cuda.set_device(dev_index)
    if not use_cuda and a.model == "resnet50" and not os.environ.get("SHIPYARD_ALLOW_CPU_RESNET50"):
        # a GPU recipe scheduled on a pool without GPUs (virtual slots): ResNet-50 at this batch size would run for hours on CPU threads
        if rank == 0:
            print(json.dumps({"error": "no GPU visible to this task: use the -CPU recipe variant (--model tiny) or set SHIPYARD_ALLOW_CPU_RESNET50=1",
                              "world": world, "model": a.model}), flush=True)
        sys.exit(2)
    torch.manual_seed(1234)
    session = os.environ.get("SHIPYARD_COLL_SESSION", f"pytorch-gpu-{os.getppid()}") + "-train"
    comm = Communicator(rank, world, session, dev_index, heap_bytes=(1 << 30) if (use_cuda or a.model == "resnet50") else (256 << 20))
    nclass = 1000 if a.model == "resnet50" else 10
    if a.model == "lenet":
        from batch_shipyard_b200.models.lenet import lenet, synthetic_digits
        a.image = 28
        model = lenet(nclass)
        tr = FusedDataParallelTrainer(model, comm, (a.batch, 1, 28, 28), nclass, lr=a.lr, weight_decay=0.0)
        st = tr.make_stager(depth=2)
        for slot in range(2):                                    # two alternating batches of learnable synthetic digits per rank
            xs, ys = synthetic_digits(a.batch, seed=1000 * rank + slot)
            st.host_x[slot].copy_(xs); st.host_y[slot].copy_(ys)
    elif a.model == "resnet20":
        from batch_shipyard_b200.models.resnet import resnet20_cifar, synthetic_cifar as synthetic_digits
        a.image = 32
        model = resnet20_cifar(nclass)
        tr = FusedDataParallelTrainer(model, comm, (a.batch, 3, 32, 32), nclass, lr=a.lr)
        st = tr.make_stager(depth=2)
        for slot in range(2):
            xs, ys = synthetic_digits(a.batch, seed=1000 * rank + slot)
            st.host_x[slot].copy_(xs); st.host_y[slot].copy_(ys)
    else:
        model = resnet50() if a.model == "resnet50" else resnet_tiny(nclass)
        tr = FusedDataParallelTrainer(model, comm, (a.batch, 3, a.image, a.image), nclass, lr=a.lr)
        st = tr.make_stager()
        st.fill_synthetic(seed=rank)
        for hy in st.host_y:
            hy.remainder_(nclass)
    st.prefetch(0); st.run_step(0); st.read_loss(0)          # first batch on the device before capture
    tr.prepare(warmup=2)
    t0 = time.time()
    losses = []
    st.prefetch(0)
    fresh = a.model in ("lenet", "resnet20") and not use_cuda           # CPU pools: a new batch of synthetic digits every step (the host buffers are plain memory)
    for i in range(a.steps):
        st.run_step(i % 2)
        if fresh:
            xs, ys = synthetic_digits(a.batch, seed=1000 * rank + 2 + i)
            st.host_x[(i + 1) % 2].copy_(xs); st.host_y[(i + 1) % 2].copy_(ys)
        st.prefetch((i + 1) % 2)
        losses.append(st.read_loss(i % 2))
    dt = time.time() - t0
    comm.check_status()
    extra = {}
    if a.model in ("lenet", "resnet20"):
        xs, ys = synthetic_digits(512, seed=987654)          # held-out digits, the same on every rank
        with torch.no_grad():
            model.eval()
            xt = (xs.to(tr.dev).float() / 255.0).permute(0, 3, 1, 2).to(tr.static_x.dtype)
            extra["test_accuracy"] = round(float((model(xt).float().argmax(1).cpu() == ys).float().mean()), 4)
    if a.eval_batches > 0:
        extra["eval"] = tr.evaluate(*_held_out(a, rank, nclass), batch=a.batch)
    if rank == 0:
        print(json.dumps({"model": a.model, "images_per_sec": round(a.batch * world * a.steps / dt, 1), "world": world, "steps": a.steps,
                          "first_loss": round(losses[0], 4), "last_loss": round(losses[-1], 4), "transport": comm.transport,
                          "own_kernels_per_step": tr.kernels_per_step, **extra}), flush=True)
    comm.close()


if __name__ == "__main__":
    main()
