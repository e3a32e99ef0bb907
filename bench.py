#!/usr/bin/env python3
"""Headline benchmark: PyTorch-GPU recipe retarget, ResNet-50 training images/sec.

Usage: ``python bench.py --gpus N --steps K --warmup W`` (N>1 under torchrun, one
rank per GPU).  Prints ONE JSON line on rank 0.

* ``value``      device-timed throughput of the captured training step (forward +
                 backward + fused all-reduce/SGD/all-gather kernel), CUDA events,
                 barrier + synchronize on both sides, max over ranks.
* ``e2e``        the same metric through the public API with, every step, the H2D
                 copy of that step's uint8 batch from pinned host memory and the
                 D2H read of the loss.
* ``baseline_same_run``  stock PyTorch (torchvision + DDP/NCCL + cuDNN, zero shipyard imports: bench/stock_baseline.py) measured in
                 THIS process on THIS lease right before the shipyard arm, in two flavours (stock-eager, stock-tuned), each
                 device-timed and end to end with its own clocks; ``vs_stock_eager`` / ``vs_stock_tuned`` are value ratios.
* ``collectives`` (N > 1) 256 MB all-reduce bus bandwidth and 8 B all-reduce latency, shipyard kernels vs NCCL, same run.
* ``--dump-outputs DIR``  after the timed steps, rank 0 writes what the last captured
                 step computed as DIR/<name>.npy: ``loss``, the model ``weights`` (bf16,
                 as float32), rank 0's fp32 ``master_weights`` and the floating-point
                 module ``buffers`` (BatchNorm running statistics).  Weight vectors over
                 4 Mi elements are reduced to the same fixed, seeded sample of positions.
                 Inputs and initial weights are seeded, so two builds can be compared
                 output for output.
* ``--impl reference``  the unmodified reference cannot be installed offline
                 (no setup.py/pyproject; imports azure.* at module load) -> prints
                 ``{"impl": "reference", "unavailable": ...}``.
* ``--impl nccl-baseline``  the bar BASELINE.md defines: torchvision resnet50 +
                 DDP/NCCL + SGD, bf16 autocast, channels_last (not our code path).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="shipyard", choices=["shipyard", "reference", "nccl-baseline"])
    ap.add_argument("--batch", type=int, default=int(os.environ.get("SHIPYARD_BENCH_BATCH", "256")), help="per-GPU batch")
    ap.add_argument("--model", default="resnet50")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-baseline", action="store_true", help="skip the same-run stock-PyTorch arms (bench/stock_baseline.py)")
    ap.add_argument("--no-coll", action="store_true", help="skip the same-run collective block (N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "shipyard":
        ap.error("--dump-outputs needs --impl shipyard")
    return args


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (profiling recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int = 0):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def dist_setup(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        args.gpus = world
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local


def max_over_ranks(x: float, world: int, dev) -> float:
    import torch
    import torch.distributed as dist
    if world == 1:
        return x
    t = torch.tensor([x], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier(world):
    import torch
    import torch.distributed as dist
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def timed(fn_step, steps: int, world: int, dev) -> float:
    """ms per step: barrier+sync, CUDA events around exactly `steps` steps, max over ranks."""
    import torch
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn_step(i)
    e1.record()
    e1.synchronize()
    barrier(world)
    ms = e0.elapsed_time(e1)
    return max_over_ranks(ms, world, dev) / steps


def run_shipyard(args, rank, world, local):
    import torch
    from batch_shipyard_b200.models.resnet import resnet50, resnet_tiny
    from batch_shipyard_b200.ops.coll import Communicator
    from batch_shipyard_b200.parallel.ddp import FusedDataParallelTrainer

    dev = torch.device("cuda", local)
    B = args.batch
    baselines = None
    if not args.no_baseline and args.model == "resnet50":
        sys.path.insert(0, os.path.join(ROOT, "bench"))
        import stock_baseline
        baselines = stock_baseline.run_both(B, args.steps, max(3, args.warmup), rank, world, local, lambda: ClockSampler(local))
    torch.manual_seed(1234)
    torch.backends.cudnn.benchmark = True
    comm = Communicator(rank, world, session=f"bench-{os.environ.get('MASTER_PORT', '0')}-{os.getppid() if world > 1 else os.getpid()}",
                        device=local, heap_bytes=1 << 30)
    model = resnet50() if args.model == "resnet50" else resnet_tiny(1000)
    tr = FusedDataParallelTrainer(model, comm, (B, 3, 224, 224), 1000, lr=0.1, momentum=0.9, weight_decay=1e-4,
                                  use_graph=not args.no_graph)
    g = torch.Generator(device="cpu").manual_seed(7 + rank)
    tr.load_images_u8(torch.randint(0, 256, (B, 224, 224, 3), dtype=torch.uint8, generator=g).to(dev),
                      torch.randint(0, 1000, (B,), generator=g).to(dev))
    tr.prepare(warmup=max(3, args.warmup))
    # --- device-timed captured step ------------------------------------------
    for _ in range(args.warmup):
        tr.step()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms = timed(lambda i: tr.step(), args.steps, world, dev)
    clocks = sampler.stop() if rank == 0 else {}
    comm.check_status()
    if args.dump_outputs and rank == 0:
        _dump_outputs(args.dump_outputs, tr)
    loss_dev = float(tr.static_loss)
    # --- end-to-end through the public API: pinned uint8 -> H2D -> convert -> step -> loss D2H
    e2e = None
    if not args.no_e2e:
        st = tr.make_stager(depth=2)
        st.fill_synthetic(seed=11 + rank)
        for i in range(max(3, args.warmup)):
            st.prefetch(i % 2); st.run_step(i % 2); st.read_loss(i % 2)
        losses = []

        def e2e_step(i):
            slot = i % 2
            if i == 0:
                st.prefetch(slot)
            st.run_step(slot)
            if i + 1 < args.steps:
                st.prefetch((i + 1) % 2)      # next batch's H2D overlaps this step's compute
            if i > 0:
                losses.append(st.read_loss((i - 1) % 2))   # D2H read of the previous step's loss

        ms_e2e = timed(e2e_step, args.steps, world, dev)
        losses.append(st.read_loss((args.steps - 1) % 2))
        e2e = {"value": round(B * world / (ms_e2e / 1e3), 2), "unit": "images/sec", "ms_per_step": round(ms_e2e, 3),
               "h2d_bytes_per_step": st.h2d_bytes, "d2h_bytes_per_step": st.d2h_bytes,
               "last_loss": round(losses[-1], 4)}
        st.close()
        e2e["input_staging"] = st.staging_summary_cached
    comm.check_status()
    if os.environ.get("SHIPYARD_BENCH_RERACE"):
        # diagnostic: run the dispatcher's race again AFTER the benchmark for the first shapes and print both tables
        from batch_shipyard_b200.ops import conv as _cv
        import torch.nn.functional as _F   # noqa: F401
        for key in list(_cv._PLANS)[:int(os.environ["SHIPYARD_BENCH_RERACE"])]:
            n_, cin, h, w_, cout, k, stride = key
            xx = (torch.randn(n_, cin, h, w_, device=dev) * 0.5).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
            ww = (torch.randn(cout, cin, k, k, device=dev) * 0.05).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
            again = _cv._autotune(xx, ww, stride)
            print(json.dumps({"rerace": "x".join(map(str, key)), "first": _cv._PLANS[key].timings_us, "again": again.timings_us}), file=sys.stderr)
    own = tr.kernels_per_step
    out = {
        "metric": "resnet50_train_images_per_sec", "value": round(B * world / (ms / 1e3), 2), "unit": "images/sec",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "impl": "shipyard",
        "config": {"model": args.model, "global_batch": B * world, "per_gpu_batch": B, "image": "3x224x224",
                   "seq_len": None, "parallelism": f"dp{world}", "optimizer": "sgd-momentum (fp32 master, sharded)",
                   "l2_policy": "per-step working set (activations) >> 126 MB L2; no explicit flush",
                   "cuda_graph": not args.no_graph, "collective_transport": comm.transport,
                   "nvls_multicast": comm.has_multicast, "conv_dispatch": _conv_summary()},
        "clocks": clocks, "e2e": e2e,
        "gpu_launches": own * args.steps + (0 if args.no_e2e else 0),
        "own_kernels_per_step": own, "loss": round(loss_dev, 4),
    }
    base = _baseline_number(world)
    if base:
        out["vs_baseline"] = round(out["value"] / base, 4)
    if baselines is not None:
        out["baseline_same_run"] = baselines
        for key, name in (("vs_stock_eager", "stock_eager"), ("vs_stock_tuned", "stock_tuned"), ("vs_stock_compiled", "stock_compiled")):
            b = baselines.get(name) or {}
            if b.get("value"):
                out[key] = {"device_timed": round(out["value"] / b["value"], 4),
                            "e2e": round(e2e["value"] / b["e2e"]["value"], 4) if (e2e and b.get("e2e", {}).get("value")) else None}
    if world > 1 and not args.no_coll:
        try:
            out["collectives"] = _collective_block(comm, rank, world, dev)
        except Exception as e:  # noqa: BLE001 - secondary block: never take the headline down
            out["collectives"] = {"error": f"{type(e).__name__}: {e}"[:200]}
    comm.close()
    return out


DUMP_SAMPLE = 4 << 20          # elements kept of each weight vector: 2 x 16 MB of float32


def _dump_outputs(out_dir: str, tr) -> None:
    """Writes what the last training step left for the caller (see --dump-outputs) as float32 .npy files."""
    import numpy as np
    import torch
    flat = tr.flat
    total = flat.params.numel()
    pos = None
    if total > DUMP_SAMPLE:
        pos = torch.randperm(total, generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
    lo, cnt = flat.shard
    in_shard = torch.arange(lo, lo + cnt) if pos is None else pos[(pos >= lo) & (pos < lo + cnt)]
    weights = flat.params.float().cpu()
    arrays = {
        "loss": tr.static_loss.detach().float().cpu().reshape(1),
        "weights": weights if pos is None else weights[pos],
        "master_weights": flat.master.float().cpu()[in_shard - lo],
        "buffers": torch.cat([b.detach().float().cpu().reshape(-1) for b in tr.model.buffers() if b.is_floating_point()]),
    }
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy().astype(np.float32))


def _collective_block(comm, rank, world, dev) -> dict:
    """A number the collectives actually limit: 256 MB fp32 all-reduce bus bandwidth and 8 B all-reduce latency, shipyard kernels
    (symmetric buffers, in place) vs NCCL through torch.distributed on the same stream, device-timed, max over ranks."""
    import torch
    import torch.distributed as dist

    def time_us(fn, iters, warm):
        for _ in range(warm):
            fn()
        barrier(world)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record(); e1.synchronize()
        return max_over_ranks(e0.elapsed_time(e1) * 1e3 / iters, world, dev)

    out = {}
    nv = _NvlinkCounters(dev.index if dev.index is not None else 0)
    for label, nbytes, iters, warm in (("allreduce_256MB", 256 << 20, 20, 5), ("allreduce_8B", 8, 200, 20)):
        n = nbytes // 4
        sym = comm.alloc(n, torch.float32); sym.fill_(1.0)
        plain = torch.ones(n, dtype=torch.float32, device=dev)
        c0 = nv.read()
        ours = time_us(lambda: comm.all_reduce(sym, sym, scale=1.0 / world), iters, warm)
        c1 = nv.read()
        nccl = time_us(lambda: dist.all_reduce(plain, op=dist.ReduceOp.AVG), iters, warm)
        c2 = nv.read()
        row = {"shipyard_us": round(ours, 2), "nccl_us": round(nccl, 2), "speedup": round(nccl / ours, 3)}
        if c0 and c1 and c2 and nbytes >= (1 << 20):
            # NVML NVLink data counters of this GPU (KiB) over the warm-up + timed calls: bytes that really crossed the links per call
            calls = iters + warm
            row["nvlink_counters_rank0"] = {
                "shipyard_tx_mb_per_call": round((c1[0] - c0[0]) / 1024.0 / calls, 1), "shipyard_rx_mb_per_call": round((c1[1] - c0[1]) / 1024.0 / calls, 1),
                "nccl_tx_mb_per_call": round((c2[0] - c1[0]) / 1024.0 / calls, 1), "nccl_rx_mb_per_call": round((c2[1] - c1[1]) / 1024.0 / calls, 1),
                "message_mb": nbytes >> 20, "note": "two-shot through the switch moves ~ message x (N-1)/N out and in per GPU; in-switch reduction (NVLS) shows as rx ~ message/N"}
        if nbytes >= (1 << 20):
            f = 2.0 * (world - 1) / world * nbytes
            row["shipyard_busbw_gbs"] = round(f / ours / 1e3, 1); row["nccl_busbw_gbs"] = round(f / nccl / 1e3, 1)
            row["frac_of_770gbs_link"] = round(f / ours / 1e3 / 770.0, 3)
        out[label] = row
    comm.check_status()
    return out


class _NvlinkCounters:
    """NVML NVLink throughput counters (data TX / RX, KiB, summed over the links of one GPU) — the evidence that a collective's bytes
    crossed NVLink, since ncu cannot replay a cross-rank kernel."""

    def __init__(self, index: int):
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:  # noqa: BLE001
            self.h = None

    def read(self):
        if self.h is None:
            return None
        try:
            nv = self.nv
            ids = [nv.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_TX, nv.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_RX]
            vals = nv.nvmlDeviceGetFieldValues(self.h, ids)
            out = []
            for v in vals:
                if v.nvmlReturn != 0:
                    return None
                out.append(int(v.value.ullVal))
            return out
        except Exception:  # noqa: BLE001
            return None


def _conv_summary():
    """How many conv passes the dispatcher put on the tcgen05 kernels vs cuDNN (per distinct layer shape)."""
    try:
        from batch_shipyard_b200.ops import conv as _conv
        tab = _conv.plan_table()
        out = {"mode": _conv._MODE, "shapes": len(tab)}
        for pas in ("fprop", "dgrad", "wgrad"):
            out[pas + "_tc"] = sum(1 for v in tab.values() if v[pas] != "cudnn")
            out[pas + "_tc_2cta"] = sum(1 for v in tab.values() if v[pas] in ("tc2", "th2"))
            out[pas + "_halo"] = sum(1 for v in tab.values() if v[pas].startswith("th"))
        out["fprop_fused_bn_stats"] = sum(1 for v in tab.values() if v["stats"])
        out["stem"] = "tc (native/gemm/stem_s2d.inc)" if _conv.stem_native() else "cudnn"
        out["tie_band"] = _conv._TIE
        # the race itself, compact: per shape and pass [library us, best own us, winner]
        race = {}
        for key, v in tab.items():
            t = v.get("timings_us") or {}
            row = {}
            for pas in ("fprop", "dgrad", "wgrad"):
                lib = t.get(pas + "_cudnn")
                own = [x for k, x in t.items() if k.startswith(pas + "_") and "cudnn" not in k]
                row[pas] = [lib, min(own) if own else None, v[pas]]
            race[key] = row
        out["race_us"] = race
        out["halo"] = _conv.halo_state()
        if os.environ.get("SHIPYARD_CONV_PLAN_DUMP"):
            os.makedirs("gpurun_out", exist_ok=True)
            with open(os.path.join("gpurun_out", "conv_plan.json"), "w") as f:
                json.dump(tab, f, indent=1)
        return out
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def _baseline_number(world: int):
    """BASELINE.md publishes nothing for the reference; once this repo has measured the plain
    NCCL/cuDNN arm the number is recorded in bench/baseline_measured.json."""
    p = os.path.join(ROOT, "bench", "baseline_measured.json")
    try:
        with open(p) as f:
            return json.load(f).get("resnet50_images_per_sec", {}).get(str(world))
    except Exception:
        return None


def run_nccl_baseline(args, rank, world, local):
    """Plain PyTorch arm: torchvision resnet50, DDP over NCCL, SGD, bf16 autocast, channels_last."""
    import torch
    import torch.nn.functional as F
    import torchvision
    dev = torch.device("cuda", local)
    torch.manual_seed(1234)
    torch.backends.cudnn.benchmark = True
    model = torchvision.models.resnet50(weights=None).to(dev).to(memory_format=torch.channels_last)
    if world > 1:
        model = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local], gradient_as_bucket_view=True)
    opt = torch.optim.SGD(model.parameters(), lr=0.1, momentum=0.9, weight_decay=1e-4)
    B = args.batch
    x = torch.randn(B, 3, 224, 224, device=dev).contiguous(memory_format=torch.channels_last)
    y = torch.randint(0, 1000, (B,), device=dev)
    hx = torch.randint(0, 256, (B, 224, 224, 3), dtype=torch.uint8).pin_memory()
    hy = torch.randint(0, 1000, (B,), dtype=torch.int64).pin_memory()
    mean = torch.tensor([0.485, 0.456, 0.406], device=dev).view(1, 3, 1, 1)
    std = torch.tensor([0.229, 0.224, 0.225], device=dev).view(1, 3, 1, 1)

    def step(xx, yy):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            loss = F.cross_entropy(model(xx), yy)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        return loss

    for _ in range(max(3, args.warmup)):
        step(x, y)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms = timed(lambda i: step(x, y), args.steps, world, dev)
    clocks = sampler.stop() if rank == 0 else {}

    def e2e_step(i):
        dx = hx.to(dev, non_blocking=True); dy = hy.to(dev, non_blocking=True)
        xx = ((dx.permute(0, 3, 1, 2).float() / 255.0 - mean) / std).contiguous(memory_format=torch.channels_last)
        float(step(xx, dy))

    for i in range(3):
        e2e_step(i)
    ms_e2e = timed(e2e_step, args.steps, world, dev)
    return {"metric": "resnet50_train_images_per_sec", "value": round(B * world / (ms / 1e3), 2), "unit": "images/sec",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "impl": "nccl-baseline",
            "config": {"model": "torchvision.resnet50", "global_batch": B * world, "per_gpu_batch": B,
                       "parallelism": f"ddp{world}", "autocast": "bf16", "memory_format": "channels_last"},
            "clocks": clocks,
            "e2e": {"value": round(B * world / (ms_e2e / 1e3), 2), "unit": "images/sec",
                    "h2d_bytes_per_step": hx.numel() + hy.numel() * 8, "d2h_bytes_per_step": 4},
            "gpu_launches": 0}


def main():
    args = parse()
    if args.impl == "reference":
        print(json.dumps({"impl": "reference", "unavailable":
                          "Azure/batch-shipyard has no setup.py/pyproject (pip cannot install it), imports azure.batch at "
                          "module load (SDK absent, no network) and contains no training/collective code to time"}))
        return 0
    import torch
    if not torch.cuda.is_available():
        print(json.dumps({"impl": args.impl, "unavailable": "no CUDA device visible"}))
        return 0
    rank, world, local = dist_setup(args)
    out = run_shipyard(args, rank, world, local) if args.impl == "shipyard" else run_nccl_baseline(args, rank, world, local)
    if rank == 0:
        print(json.dumps(out), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
