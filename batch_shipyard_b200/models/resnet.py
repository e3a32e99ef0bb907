"""ResNet-50 (v1.5) for the PyTorch-GPU recipe retarget.

The reference's ``recipes/PyTorch-GPU`` only launches a user container running
stock PyTorch (/root/reference/recipes/PyTorch-GPU/config/jobs.yaml:1-8); the
north star retargets it to multi-instance ResNet-50.  This is our own
implementation (not torchvision): NHWC/bf16 end to end, parameters are views
into ONE flat symmetric buffer so the fused all-reduce + SGD kernel
(``ops.coll.Communicator.fused_allreduce_sgd``) updates the whole model in a
single launch.
"""
from __future__ import annotations

import math
from typing import Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from ..ops import conv as _conv
from ..ops import fused as _fused
from ..ops import gemm as _gemm


import os as _os0

# Residual-gradient fusion is ON by default since round 2: gradients match fp32 torchvision within the bf16 noise floor
# (tests/test_gpu_resnet_parity.py::test_resnet50_residual_gradient_fusion_matches_torchvision) and the step is ~0.3 ms shorter
# (gpurun_out/c6_bench_dual.json: 20.25 ms vs 20.53 ms in the same call).  SHIPYARD_BN_DUAL=0 restores the autograd add kernels.
_BN_DUAL = [_os0.environ.get("SHIPYARD_BN_DUAL", "1") not in ("0", "", "off", "false")]


def set_bn_dual(on: bool) -> None:
    """Residual-gradient fusion (two-handle block outputs) on / off; read at forward time."""
    _BN_DUAL[0] = bool(on)


class ConvBN(nn.Module):
    """conv (no bias) + train-mode BatchNorm (+ residual add) (+ ReLU)."""

    def __init__(self, cin: int, cout: int, k: int, stride: int = 1, relu: bool = True, zero_gamma: bool = False):
        super().__init__()
        self.cin, self.cout, self.k, self.stride, self.relu = cin, cout, k, stride, relu
        self.weight = nn.Parameter(torch.empty(cout, cin, k, k))
        nn.init.kaiming_normal_(self.weight, mode="fan_out", nonlinearity="relu")
        self.gamma = nn.Parameter(torch.zeros(cout) if zero_gamma else torch.ones(cout))
        self.beta = nn.Parameter(torch.zeros(cout))
        self.register_buffer("running_mean", torch.zeros(cout, dtype=torch.float32))
        self.register_buffer("running_var", torch.ones(cout, dtype=torch.float32))
        self.momentum, self.eps = 0.1, 1e-5
        import os as _os
        self.use_tc_gemm = not _os.environ.get("SHIPYARD_NO_TC_GEMM")     # off: plain cuDNN path, no dispatcher

    def forward(self, x: torch.Tensor, residual: Optional[torch.Tensor] = None, dual: bool = False):
        fast = x.is_cuda and self.training and x.dtype == torch.bfloat16
        stats = None
        if fast and self.k in (1, 3) and self.use_tc_gemm:
            # dispatcher: per shape and per pass the faster of the tcgen05 implicit-GEMM kernels and cuDNN (measured once,
            # during the eager warm-up step); BN statistics come from the epilogue when the tcgen05 fprop wins
            y, stats = _conv.conv_bn_input(x, self.weight, self.stride)
        elif self.k == 7 and x.shape[1] == 16:
            # space-to-depth stem: the 7x7/s2/p3 conv as a dense 4x4/s1 conv over the 16-channel s2d input
            w2 = _fused.stem_weight_s2d(self.weight).contiguous(memory_format=torch.channels_last)
            if fast and self.use_tc_gemm and self.cout == 64 and _conv.stem_native() and _gemm.stem_s2d_ok(x, w2):
                # own tcgen05 kernels (fprop with BN statistics in the epilogue, wgrad); cuDNN needs ~5x longer on C = 16
                y, stats = _gemm.stem_conv_s2d(x, w2, True)
            else:
                y = F.conv2d(x, w2)
        else:
            y = F.conv2d(x, self.weight, None, self.stride, self.k // 2)
        if fast:
            # one fused stats + apply(+residual)(+ReLU) pair instead of BN / add / ReLU kernels;
            # no eager fallback on GPU: a missing extension must fail loudly
            return _fused.fused_bn_act(y, self.gamma, self.beta, residual, self.running_mean, self.running_var,
                                       self.relu, self.eps, self.momentum, stats=stats, dual=dual)
        y = F.batch_norm(y.float(), self.running_mean, self.running_var, self.gamma.float(), self.beta.float(),
                         self.training, self.momentum, self.eps).to(y.dtype)
        if residual is not None:
            y = y + residual
        return F.relu(y) if self.relu else y


class Bottleneck(nn.Module):
    expansion = 4

    def __init__(self, cin: int, width: int, stride: int):
        super().__init__()
        cout = width * self.expansion
        self.c1 = ConvBN(cin, width, 1)
        self.c2 = ConvBN(width, width, 3, stride)          # v1.5: stride on the 3x3
        self.c3 = ConvBN(width, cout, 1, relu=True, zero_gamma=True)
        self.down = ConvBN(cin, cout, 1, stride, relu=False) if (stride != 1 or cin != cout) else None

    def forward(self, x):
        # SHIPYARD_BN_DUAL: the block output travels as two handles of one tensor (ops.fused.fused_bn_act(dual=True)); the next
        # block gives one to its first convolution and one to its residual input, so the two gradients meet inside the BN
        # backward kernels of THIS block instead of in a separate add kernel (12 of the 16 blocks of ResNet-50).
        xm, xa = x if isinstance(x, tuple) else (x, x)
        idt = xa if self.down is None else self.down(xm)
        return self.c3(self.c2(self.c1(xm)), residual=idt, dual=_BN_DUAL[0])


class ResNet(nn.Module):
    def __init__(self, layers=(3, 4, 6, 3), num_classes: int = 1000, width: int = 64):
        super().__init__()
        self.stem = ConvBN(3, width, 7, 2)
        blocks, cin = [], width
        for i, n in enumerate(layers):
            w = width * (2 ** i)
            for j in range(n):
                blocks.append(Bottleneck(cin, w, (1 if i == 0 else 2) if j == 0 else 1))
                cin = w * Bottleneck.expansion
        self.blocks = nn.Sequential(*blocks)
        self.fc_weight = nn.Parameter(torch.empty(num_classes, cin))
        self.fc_bias = nn.Parameter(torch.zeros(num_classes))
        nn.init.kaiming_uniform_(self.fc_weight, a=math.sqrt(5))
        bound = 1 / math.sqrt(cin)
        nn.init.uniform_(self.fc_bias, -bound, bound)
        import os as _os
        self.use_tc_gemm = not _os.environ.get("SHIPYARD_NO_TC_GEMM")
        self.s2d_stem = True      # CUDA trainers feed the stem a space-to-depth input (see ops.fused.u8_to_s2d_norm)

    def forward(self, x):
        x = self.stem(x)
        fast = x.is_cuda and x.dtype == torch.bfloat16 and self.training
        x = _fused.maxpool3x3s2(x) if (fast and x.shape[1] % 8 == 0) else F.max_pool2d(x, 3, 2, 1)
        x = self.blocks(x)
        if isinstance(x, tuple):
            x = x[0]
        x = x.mean(dim=(2, 3))
        if fast and self.use_tc_gemm:
            return _gemm.linear(x, self.fc_weight, self.fc_bias)          # FC on the tcgen05 kernel (bias fused)
        return F.linear(x, self.fc_weight, self.fc_bias)


def resnet50(num_classes: int = 1000) -> ResNet:
    return ResNet((3, 4, 6, 3), num_classes)


def resnet_tiny(num_classes: int = 10) -> ResNet:
    """Two-block variant for smoke tests."""
    return ResNet((1, 1, 1, 1), num_classes, width=16)


class BasicBlock(nn.Module):
    """Two 3x3 ConvBN layers with an identity / 1x1 projection shortcut (the CIFAR ResNet block)."""

    def __init__(self, cin: int, cout: int, stride: int):
        super().__init__()
        self.c1 = ConvBN(cin, cout, 3, stride)
        self.c2 = ConvBN(cout, cout, 3, 1, relu=True, zero_gamma=True)
        self.down = ConvBN(cin, cout, 1, stride, relu=False) if (stride != 1 or cin != cout) else None

    def forward(self, x):
        idt = x if self.down is None else self.down(x)
        return self.c2(self.c1(x), residual=idt)


class ResNetCifar(nn.Module):
    """ResNet-6n+2 for 32x32 inputs (n = 3: ResNet-20): 3x3 stem, three stages of n BasicBlocks at 16 / 32 / 64 channels, global average
    pool, linear classifier — the network behind the CIFAR-10 examples of the reference's MXNet and CNTK recipes
    (/root/reference/recipes/MXNet-CPU/README.md:39-40 "cifar-10 examples run resnet")."""
    s2d_stem = False

    def __init__(self, n: int = 3, num_classes: int = 10, width: int = 16):
        super().__init__()
        self.stem = ConvBN(3, width, 3, 1)
        blocks, cin = [], width
        for i in range(3):
            for j in range(n):
                blocks.append(BasicBlock(cin, width * 2 ** i, 2 if (i > 0 and j == 0) else 1))
                cin = width * 2 ** i
        self.blocks = nn.Sequential(*blocks)
        self.fc = nn.Linear(cin, num_classes)
        for m in self.modules():                      # small channel counts: plain library convolutions, no dispatcher race
            if hasattr(m, "use_tc_gemm"):
                m.use_tc_gemm = False

    def forward(self, x):
        x = self.blocks(self.stem(x))
        return self.fc(x.mean(dim=(2, 3)).to(self.fc.weight.dtype))


def resnet20_cifar(num_classes: int = 10) -> ResNetCifar:
    return ResNetCifar(3, num_classes)


def synthetic_cifar(n: int, seed: int, num_classes: int = 10, size: int = 32):
    """CIFAR-shaped synthetic data with a learnable signal: every class is a fixed low-frequency colour pattern (seed-independent) plus
    per-sample shift, contrast jitter and pixel noise.  Returns uint8 NHWC images [n, size, size, 3] and int64 labels."""
    g0 = torch.Generator().manual_seed(4321)
    coarse = torch.rand(num_classes, 3, 4, 4, generator=g0)
    templates = F.interpolate(coarse, size=(size, size), mode="bilinear", align_corners=False)
    g = torch.Generator().manual_seed(seed)
    y = torch.randint(0, num_classes, (n,), generator=g)
    dx, dy = torch.randint(-3, 4, (n,), generator=g), torch.randint(-3, 4, (n,), generator=g)
    x = torch.stack([torch.roll(templates[int(c)], (int(a), int(b)), (1, 2)) for c, a, b in zip(y, dy, dx)])
    x = (x - 0.5) * (0.7 + 0.6 * torch.rand(n, 1, 1, 1, generator=g)) + 0.5 + 0.15 * (torch.rand(n, 3, size, size, generator=g) - 0.5)
    return (x.clamp(0, 1) * 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous(), y


def _torchvision_name_map(model: ResNet) -> dict:
    """torchvision resnet state-dict key -> (our tensor, kind) for every parameter and BN statistic of ``model``."""
    out = {}

    def cb(prefix_conv, prefix_bn, c: ConvBN):
        out[prefix_conv + ".weight"] = c.weight
        out[prefix_bn + ".weight"] = c.gamma
        out[prefix_bn + ".bias"] = c.beta
        out[prefix_bn + ".running_mean"] = c.running_mean
        out[prefix_bn + ".running_var"] = c.running_var

    cb("conv1", "bn1", model.stem)
    # our blocks are one flat Sequential; torchvision groups them into layer1..layer4, and the first block of every stage is the one
    # with a projection shortcut (the width changes by the expansion factor at every stage start)
    layers = []
    for b in model.blocks:
        if not layers or b.down is not None:
            layers.append([])
        layers[-1].append(b)
    for li, blocks in enumerate(layers):
        for j, b in enumerate(blocks):
            p = f"layer{li + 1}.{j}"
            cb(p + ".conv1", p + ".bn1", b.c1)
            cb(p + ".conv2", p + ".bn2", b.c2)
            cb(p + ".conv3", p + ".bn3", b.c3)
            if b.down is not None:
                cb(p + ".downsample.0", p + ".downsample.1", b.down)
    out["fc.weight"] = model.fc_weight
    out["fc.bias"] = model.fc_bias
    return out


def load_torchvision_state_dict(model: ResNet, sd: dict) -> ResNet:
    """Copy a torchvision ResNet (Bottleneck) state dict into ``model``: ``conv1`` / ``bn1``, ``layerX.Y.convZ`` / ``bnZ``,
    ``layerX.Y.downsample.0`` / ``.1`` and ``fc``, running statistics included (``num_batches_tracked`` is ignored).

    Raises ``KeyError`` listing the names on any unused key, missing key or shape mismatch, and changes nothing in that case.
    Call it before building a trainer: ``FusedDataParallelTrainer`` takes its fp32 master copy of the weights at construction."""
    names = _torchvision_name_map(model)
    keys = {k for k in sd if not k.endswith("num_batches_tracked")}
    unused = sorted(keys - set(names))
    missing = sorted(set(names) - keys)
    shape = sorted(k for k in keys & set(names) if tuple(sd[k].shape) != tuple(names[k].shape))
    if unused or missing or shape:
        parts = []
        if unused:
            parts.append("unused keys: " + ", ".join(unused))
        if missing:
            parts.append("missing keys: " + ", ".join(missing))
        if shape:
            parts.append("shape mismatch: " + ", ".join(f"{k} {tuple(sd[k].shape)} vs {tuple(names[k].shape)}" for k in shape))
        raise KeyError("; ".join(parts))
    with torch.no_grad():
        for k, t in names.items():
            t.copy_(sd[k].to(device=t.device, dtype=t.dtype))
    return model


def set_tc_gemm(m: nn.Module, flag: bool) -> None:
    for mod in m.modules():
        if hasattr(mod, "use_tc_gemm"):
            mod.use_tc_gemm = flag


def param_count(m: nn.Module) -> int:
    return sum(p.numel() for p in m.parameters())
