#!/usr/bin/env python3
"""ResNet-50 inference throughput on one GPU: the project's engine (parallel.infer.ResNetInference) against same-run stock arms.

Arms (all bf16, 224 x 224, the same seeded uint8 batch):
  engine          graph-captured engine, device-timed over graph replays (CUDA events) after a warm-up;
  engine_e2e      the same engine fed from pinned host uint8 batches (host-to-device copy + conversion + replay), wall clock;
  stock_graph     torchvision resnet50 in eval(), bf16, channels_last, captured in a CUDA graph (stock_* arms import nothing from
                  this project, like bench/stock_baseline.py);
  stock_compiled  the same model under torch.compile (inductor), device-timed (--no-compile skips it).
Also reported: own kernels per batch, the inference plan table (own kernel or cuDNN per layer shape), the device name and power
limit read in this call, and max |logits(engine) - logits(stock_graph)| on the same input with the same weights.
Prints one JSON line.  Usage: python bench/infer_bench.py --batch 256 [--iters 50] [--warmup 10]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _timed(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / iters / 1e3          # seconds per batch


def _device_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["max_sm_clock_mhz"] = float(q[0]), float(q[1])
    except Exception as e:  # noqa: BLE001
        info["power_limit_w"] = f"unavailable: {e}"
    return info


def stock_model(weights_sd, batch):
    """torchvision resnet50, eval, bf16, channels_last (no project imports)."""
    import torchvision
    m = torchvision.models.resnet50()
    m.load_state_dict(weights_sd)
    return m.cuda().eval().to(torch.bfloat16).to(memory_format=torch.channels_last)


def stock_input(img_u8):
    mean = torch.tensor((0.485, 0.456, 0.406), device="cuda"); std = torch.tensor((0.229, 0.224, 0.225), device="cuda")
    return ((img_u8.float() / 255.0 - mean) / std).permute(0, 3, 1, 2).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--no-compile", action="store_true")
    a = ap.parse_args()
    torch.backends.cudnn.benchmark = True
    torch.manual_seed(0)
    import torchvision
    tv = torchvision.models.resnet50()
    with torch.no_grad():
        for mod in tv.modules():
            if isinstance(mod, torch.nn.BatchNorm2d):
                mod.weight.uniform_(0.5, 1.5); mod.bias.uniform_(-0.3, 0.3)
                mod.running_mean.uniform_(-0.2, 0.2); mod.running_var.uniform_(0.5, 2.0)
    sd = tv.state_dict()
    g = torch.Generator(device="cuda").manual_seed(1)
    img = torch.randint(0, 256, (a.batch, 224, 224, 3), dtype=torch.uint8, device="cuda", generator=g)
    out = {"bench": "resnet50_inference", "batch": a.batch, **_device_info()}

    # ---- stock arms ----------------------------------------------------------------------------------------------------------
    sm = stock_model(sd, a.batch)
    xs = stock_input(img)
    with torch.no_grad():
        for _ in range(3):
            sm(xs)
        torch.cuda.synchronize()
        sg = torch.cuda.CUDAGraph()
        with torch.cuda.graph(sg):
            stock_logits = sm(xs)
    t = _timed(sg.replay, a.iters, a.warmup)
    out["stock_graph_img_s"] = round(a.batch / t, 1)
    if not a.no_compile:
        try:
            cm = torch.compile(sm)
            with torch.no_grad():
                t0 = time.time()
                for _ in range(3):
                    cm(xs)
                torch.cuda.synchronize()
                out["stock_compiled_compile_s"] = round(time.time() - t0, 1)
                t = _timed(lambda: cm(xs), a.iters, a.warmup)
            out["stock_compiled_img_s"] = round(a.batch / t, 1)
        except Exception as e:  # noqa: BLE001
            out["stock_compiled_img_s"] = f"failed: {type(e).__name__}: {str(e)[:200]}"

    # ---- engine --------------------------------------------------------------------------------------------------------------
    sys.path.insert(0, ROOT)
    from batch_shipyard_b200.models.resnet import load_torchvision_state_dict, resnet50
    from batch_shipyard_b200.ops import conv
    from batch_shipyard_b200.parallel.infer import ResNetInference, cast_for_inference
    ours = resnet50()
    load_torchvision_state_dict(ours, sd)
    cast_for_inference(ours, "cuda")
    t0 = time.time()
    eng = ResNetInference(ours, a.batch)
    out["engine_build_s"] = round(time.time() - t0, 1)
    logits = eng(img)
    out["max_abs_dlogits_vs_stock_graph"] = round(float((logits - stock_logits.float()).abs().max()), 4)
    out["max_abs_logit_stock_graph"] = round(float(stock_logits.float().abs().max()), 4)
    eng.static_u8.copy_(img)
    t = _timed(eng.graph.replay, a.iters, a.warmup)
    out["engine_img_s"] = round(a.batch / t, 1)
    # end to end: pinned host uint8 -> device (copy on its own stream, overlapped with the previous batch) -> engine
    host = [img.cpu().pin_memory() for _ in range(2)]
    dev = [torch.empty_like(img) for _ in range(2)]
    cp = torch.cuda.Stream()
    done = [torch.cuda.Event() for _ in range(2)]
    used = [torch.cuda.Event() for _ in range(2)]
    cur = torch.cuda.current_stream()
    def e2e_run(n):
        for i in range(n):
            s = i % 2
            with torch.cuda.stream(cp):
                cp.wait_event(used[s])
                dev[s].copy_(host[s], non_blocking=True)
                done[s].record(cp)
            cur.wait_event(done[s])
            eng.static_u8.copy_(dev[s])
            used[s].record(cur)
            eng.graph.replay()
        torch.cuda.synchronize()
    e2e_run(a.warmup)
    t0 = time.time()
    e2e_run(a.iters)
    out["engine_e2e_img_s"] = round(a.batch * a.iters / (time.time() - t0), 1)
    out["kernels_per_batch"] = eng.kernels_per_batch
    table = conv.infer_plan_table()
    out["own_kernel_shapes"] = sum(1 for v in table.values() if v["impl"] == "tc")
    out["plan_shapes"] = len(table)
    out["infer_plan"] = table
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
