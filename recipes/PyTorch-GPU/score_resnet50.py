#!/usr/bin/env python3
"""PyTorch-GPU recipe body: batch scoring with ResNet-50, one rank per GPU.

Every rank scores a contiguous slice of one uint8 NHWC image file (``--images``, memory-mapped) on the graph-captured inference engine
(``parallel.infer.ResNetInference``: BatchNorm folded into the tcgen05 convolution epilogue).  The host-to-device copy of the next batch
runs on the stager's copy stream while the current batch is scored (the same ``ops.stage.Stager`` tickets the training input path
uses).  Rank r writes its top-5 class indices to ``DIR/top5.rank<r>.npy``; rank 0 prints one JSON line with the whole job's rate
(wall clock, host-to-device copies included) and, when ``--labels`` is given, the top-1 / top-5 accuracy over all ranks.

``--weights`` loads a torchvision ResNet-50 state dict (``torch.load(weights_only=True)``).  Without ``--images`` a seeded synthetic
file of ``--synthetic`` images is scored, so the job runs as shipped.  On a CPU slot ``--model tiny`` runs the module's eval forward.
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.environ.get("SHIPYARD_HOME") or os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from batch_shipyard_b200.models.resnet import load_torchvision_state_dict, resnet50, resnet_tiny  # noqa: E402
from batch_shipyard_b200.ops.coll import Communicator  # noqa: E402


def _synthetic(out_dir, n, image, classes, rank):
    """Seeded uint8 NHWC images + labels, written once (rank 0, atomic rename) and memory-mapped by every rank."""
    path, lpath = os.path.join(out_dir, "synthetic_images.npy"), os.path.join(out_dir, "synthetic_labels.npy")
    if rank == 0 and not (os.path.exists(path) and np.load(path, mmap_mode="r").shape == (n, image, image, 3)):
        rng = np.random.default_rng(20261017)
        for p, arr in ((path, rng.integers(0, 256, (n, image, image, 3), dtype=np.uint8)),
                       (lpath, rng.integers(0, classes, (n,), dtype=np.int64))):
            tmp = p + ".tmp%d" % os.getpid()
            with open(tmp, "wb") as f:
                np.save(f, arr)
            os.replace(tmp, p)
    return path, lpath


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", help="uint8 NHWC .npy [N, H, W, 3] (memory-mapped)")
    ap.add_argument("--labels", help="int64 .npy [N] (optional: top-1 / top-5 accuracy)")
    ap.add_argument("--weights", help="torchvision ResNet state dict (torch.save of model.state_dict())")
    ap.add_argument("--batch", type=int, default=256, help="per-GPU batch")
    ap.add_argument("--out", default="score_out", help="directory for top5.rank<r>.npy")
    ap.add_argument("--synthetic", type=int, default=4096, help="without --images: score this many seeded synthetic images")
    ap.add_argument("--image", type=int, default=224, help="image size of the synthetic file")
    ap.add_argument("--model", default="resnet50", choices=["resnet50", "tiny"])
    a = ap.parse_args()
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    gpu = os.environ.get("SHIPYARD_GPU", os.environ.get("LOCAL_RANK", "0"))
    use_cuda = torch.cuda.is_available() and gpu not in ("", "-1")
    dev_index = int(gpu) % max(1, torch.cuda.device_count()) if use_cuda else None
    if use_cuda:
        torch.cuda.set_device(dev_index)
    if not use_cuda and a.model == "resnet50" and not os.environ.get("SHIPYARD_ALLOW_CPU_RESNET50"):
        if rank == 0:
            print(json.dumps({"error": "no GPU visible to this task: use --model tiny on CPU slots or set SHIPYARD_ALLOW_CPU_RESNET50=1",
                              "world": world, "model": a.model}), flush=True)
        sys.exit(2)
    os.makedirs(a.out, exist_ok=True)
    session = os.environ.get("SHIPYARD_COLL_SESSION", f"pytorch-gpu-{os.getppid()}") + "-score"
    comm = Communicator(rank, world, session, dev_index, heap_bytes=1 << 20)
    nclass = 1000 if a.model == "resnet50" else 10
    images, labels = a.images, a.labels
    if images is None:
        images, labels = _synthetic(a.out, a.synthetic, a.image, nclass, rank)
    comm.barrier()                                                      # the synthetic file is complete before anyone maps it
    x_all = np.load(images, mmap_mode="r")
    y_all = np.load(labels, mmap_mode="r") if labels else None
    n_all, h, w, c = x_all.shape
    assert c == 3 and x_all.dtype == np.uint8, (x_all.dtype, x_all.shape)
    lo, hi = n_all * rank // world, n_all * (rank + 1) // world

    torch.manual_seed(0)
    model = resnet50(nclass) if a.model == "resnet50" else resnet_tiny(nclass)
    if a.weights:
        load_torchvision_state_dict(model, torch.load(a.weights, map_location="cpu", weights_only=True))
    model.eval()
    top5 = np.zeros((hi - lo, 5), dtype=np.int64)
    comm.barrier()
    t0 = time.time()
    if use_cuda:
        from batch_shipyard_b200.ops.stage import Stager
        from batch_shipyard_b200.parallel.infer import ResNetInference, cast_for_inference
        dev = torch.device("cuda", dev_index)
        cast_for_inference(model, dev)
        eng = ResNetInference(model, a.batch, image_size=h)
        comm.barrier()
        t0 = time.time()                                                # the rate covers scoring, not the one-time engine build
        bs = a.batch
        host = [torch.empty((bs, h, w, 3), dtype=torch.uint8, pin_memory=True) for _ in range(2)]
        devb = [torch.empty((bs, h, w, 3), dtype=torch.uint8, device=dev) for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]
        used = [False, False]
        stager = Stager(dev_index, arena_bytes=8 << 20, concurrency=1)
        tickets = [None, None]
        starts = list(range(lo, hi, bs))

        def prefetch(i):
            s, b0 = i % 2, starts[i]
            n = min(bs, hi - b0)
            if tickets[s] is not None:                                   # the previous copy out of this pinned slot has finished
                stager.wait(tickets[s]); stager.release(tickets[s]); tickets[s] = None
            host[s][:n].numpy()[...] = x_all[b0:b0 + n]
            # the copy stream waits until the batch that last used the device slot has been read by the engine
            tickets[s] = stager.submit_pinned(host[s].data_ptr(), n * h * w * 3, devb[s].data_ptr(),
                                              consumed[s].cuda_event if used[s] else 0)
            used[s] = True

        cur = torch.cuda.current_stream(dev)
        if starts:
            prefetch(0)
        for i, b0 in enumerate(starts):
            s, n = i % 2, min(bs, hi - starts[i])
            stager.stream_wait(tickets[s], cur.cuda_stream)             # scoring waits for its batch's copy, the host does not
            logits = eng(devb[s][:n])
            consumed[s].record(cur)
            if i + 1 < len(starts):
                prefetch(i + 1)                                         # overlaps the batch just enqueued
            top5[b0 - lo:b0 - lo + n] = logits.topk(5, dim=1).indices.cpu().numpy()
        torch.cuda.synchronize(dev)
        for t in tickets:
            if t is not None:
                stager.wait(t); stager.release(t)
        stager.close()
        kernels = eng.kernels_per_batch
    else:
        with torch.no_grad():
            for b0 in range(lo, hi, a.batch):
                xb = torch.from_numpy(np.ascontiguousarray(x_all[b0:min(hi, b0 + a.batch)]))
                logits = model((xb.float() / 255.0).permute(0, 3, 1, 2))
                top5[b0 - lo:b0 - lo + xb.shape[0]] = logits.topk(min(5, logits.shape[1]), dim=1).indices.numpy()
        kernels = 0
    np.save(os.path.join(a.out, f"top5.rank{rank}.npy"), top5)
    sums = comm.alloc(3, torch.float64)
    local = [float(hi - lo), 0.0, 0.0]
    if y_all is not None:
        yy = np.asarray(y_all[lo:hi]).reshape(-1, 1)
        local[1], local[2] = float((top5[:, :1] == yy).sum()), float((top5 == yy).any(axis=1).sum())
    sums.copy_(torch.tensor(local, dtype=torch.float64).to(sums.device))
    comm.all_reduce(sums)
    if use_cuda:
        torch.cuda.synchronize()
    dt = time.time() - t0
    tot = sums.cpu().tolist()
    comm.check_status()
    if rank == 0:
        out = {"model": a.model, "images": int(tot[0]), "images_per_sec": round(tot[0] / dt, 1), "world": world,
               "batch": a.batch, "transport": comm.transport, "own_kernels_per_batch": kernels, "out": os.path.abspath(a.out)}
        if y_all is not None:
            out["top1"], out["top5"] = round(tot[1] / max(1.0, tot[0]), 4), round(tot[2] / max(1.0, tot[0]), 4)
        print(json.dumps(out), flush=True)
    comm.close()


if __name__ == "__main__":
    main()
