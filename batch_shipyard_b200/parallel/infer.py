"""ResNet inference on the project's sm_100a kernels: BatchNorm folded into the convolution epilogue, one CUDA graph per batch.

``ResNetInference(model, batch)`` serves ``ResNet`` (resnet50, resnet_tiny) and ``ResNetCifar`` (resnet20).  It walks the model's
modules itself and never calls ``forward()``, so the training path is untouched.  One call converts a static uint8 NHWC batch:

1. input conversion with the kernels training uses (``u8_to_s2d_norm`` for the space-to-depth stem, ``u8_to_bf16_norm`` otherwise),
   so evaluation sees exactly what training saw;
2. ``bn_fold``: one launch turns every BN layer's current gamma / beta / running statistics into fp32 scale / shift;
3. the stem (own ``stem_s2d_fprop`` or cuDNN), then ``bn_infer_apply`` (+ ReLU);
4. the index-free max-pool;
5. every block: ``down`` first, then the last convolution with ``residual=``; each convolution runs conv + BN (+ residual) (+ ReLU)
   either as one tcgen05 kernel with the affine epilogue or as cuDNN + ``bn_infer_apply``, whichever the per-shape race of
   ``ops.conv.infer_plan_for`` chose;
6. the mean pool and the FC GEMM with the bias fused in its epilogue.

The race runs in an eager warm-up at construction; the whole call is then captured as one CUDA graph.  The engine reads the
parameters and statistics in place and never writes them, nor the optimizer state or ``model.training``.
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn.functional as F

from ..ops import conv as _conv
from ..ops import fused as _fused
from ..ops import gemm as _gemm


def cast_for_inference(model: torch.nn.Module, device) -> torch.nn.Module:
    """Put a model in the form the engine reads, in place: parameters bf16 on ``device`` (convolution weights channels_last, the KRSC
    layout of the kernels), BatchNorm running statistics fp32 on ``device``.  (``model.to(torch.bfloat16)`` would also cast the
    statistics.)"""
    model.to(device)
    for p in model.parameters():
        p.data = p.data.to(torch.bfloat16)
        if p.dim() == 4:
            p.data = p.data.contiguous(memory_format=torch.channels_last)
    for b in model.buffers():
        if b.is_floating_point():
            b.data = b.data.float()
    return model


def _launches() -> int:
    return _fused.launch_count() + _gemm.launch_count()


class ResNetInference:
    """Graph-captured inference of a ResNet at a fixed batch size; ``eng(images_u8)`` returns fp32 logits ``[n, classes]``.

    The parameters must be bf16 and the running statistics fp32 on a CUDA device (a trainer's model is; ``cast_for_inference``
    prepares any other).  The fold table holds raw pointers to gamma / beta / running statistics, and the
    graph reads the convolution and FC weights at their addresses: rebuild the engine if the parameters or buffers are moved to new
    storage (``model.to(...)``, re-creating a trainer).  Updating them in place (an optimizer step) needs no rebuild."""

    def __init__(self, model: torch.nn.Module, batch: int, image_size: Optional[int] = None, use_graph: bool = True):
        from ..models.resnet import Bottleneck, BasicBlock, ResNet, ResNetCifar
        if not isinstance(model, (ResNet, ResNetCifar)):
            raise TypeError(f"ResNetInference serves ResNet / ResNetCifar, not {type(model).__name__}")
        p0 = next(model.parameters())
        if not (p0.is_cuda and all(p.dtype == torch.bfloat16 for p in model.parameters())):
            raise ValueError("ResNetInference needs bf16 parameters on a CUDA device")
        self.model, self.batch, self.dev = model, int(batch), p0.device
        self.cifar = isinstance(model, ResNetCifar)
        size = int(image_size or (32 if self.cifar else 224))
        self.image_size = size
        self.s2d = bool(getattr(model, "s2d_stem", False)) and not self.cifar and size % 2 == 0
        # every ConvBN in execution order; the fold table follows the same order
        self.blocks = []
        convs = [model.stem]
        for b in model.blocks:
            if isinstance(b, Bottleneck):
                self.blocks.append(("bottleneck", b))
                convs += [c for c in (b.down, b.c1, b.c2, b.c3) if c is not None]
            elif isinstance(b, BasicBlock):
                self.blocks.append(("basic", b))
                convs += [c for c in (b.down, b.c1, b.c2) if c is not None]
            else:
                raise TypeError(f"unsupported block {type(b).__name__}")
        self.convs = convs
        self.fold = _fused.BnFoldTable([(c.gamma, c.beta, c.running_mean, c.running_var, c.eps) for c in convs], self.dev)
        self._idx = {id(c): i for i, c in enumerate(convs)}
        if self.cifar:
            self.fc_w, self.fc_b = model.fc.weight, model.fc.bias
        else:
            self.fc_w, self.fc_b = model.fc_weight, model.fc_bias
        self.num_classes = self.fc_w.shape[0]
        n = self.batch
        self.static_u8 = torch.zeros((n, size, size, 3), dtype=torch.uint8, device=self.dev)
        if self.s2d:
            self._x_store = torch.zeros((n, size // 2 + 3, size // 2 + 3, 16), dtype=torch.bfloat16, device=self.dev)
        else:
            self._x_store = torch.zeros((n, size, size, 3), dtype=torch.bfloat16, device=self.dev)
        self.static_logits = torch.zeros((n, self.num_classes), dtype=torch.float32, device=self.dev)
        self.graph = None
        self.kernels_per_batch = 0
        # eager warm-up: races every layer shape (ops.conv.infer_plan_for) and lets cuDNN pick its algorithms
        with torch.no_grad():
            s = torch.cuda.Stream(self.dev)
            s.wait_stream(torch.cuda.current_stream(self.dev))
            with torch.cuda.stream(s):
                self._forward()
                before = _launches()
                self._forward()
                self.kernels_per_batch = _launches() - before
            torch.cuda.current_stream(self.dev).wait_stream(s)
            torch.cuda.synchronize(self.dev)
            if use_graph:
                self.graph = torch.cuda.CUDAGraph()
                before = _launches()
                with torch.cuda.graph(self.graph):
                    self._forward()
                self.kernels_per_batch = _launches() - before
                torch.cuda.synchronize(self.dev)

    # -- one batch on the static buffers ---------------------------------------------------------------------------------------
    def _bn(self, c, y, residual=None, relu=None):
        i = self._idx[id(c)]
        return _fused.bn_infer_apply(y, self.fold.scale[i], self.fold.shift[i], residual, c.relu if relu is None else relu, out=y)

    def _conv(self, c, x, residual=None):
        i = self._idx[id(c)]
        return _conv.conv_bn_infer(x, c.weight, self.fold.scale[i], self.fold.shift[i], c.stride, residual=residual, relu=c.relu,
                                   use_tc=bool(c.use_tc_gemm) and c.k in (1, 3))

    def _stem(self, x):
        c = self.model.stem
        if self.s2d:
            w2 = _fused.stem_weight_s2d(c.weight).contiguous(memory_format=torch.channels_last)
            if c.use_tc_gemm and c.cout == 64 and _conv.stem_native() and _gemm.stem_s2d_ok(x, w2):
                y = _gemm.stem_s2d_fprop(x, w2)
            else:
                y = F.conv2d(x, w2)
        else:
            y = F.conv2d(x, c.weight, None, c.stride, c.k // 2)
        if not y.is_contiguous(memory_format=torch.channels_last):
            y = y.contiguous(memory_format=torch.channels_last)
        return self._bn(c, y)

    def _forward(self) -> None:
        if self.s2d:
            _fused.u8_to_s2d_norm(self.static_u8, self._x_store)
        else:
            _fused.u8_to_bf16_norm(self.static_u8, self._x_store)
        _fused.bn_fold(self.fold)
        x = self._stem(self._x_store.permute(0, 3, 1, 2))
        if not self.cifar:
            x = _fused.maxpool3x3s2_infer(x)
        for kind, b in self.blocks:
            idt = x if b.down is None else self._conv(b.down, x)
            if kind == "bottleneck":
                y = self._conv(b.c2, self._conv(b.c1, x))
                x = self._conv(b.c3, y, residual=idt)
            else:
                x = self._conv(b.c2, self._conv(b.c1, x), residual=idt)
        pooled = x.mean(dim=(2, 3))
        logits = _gemm.gemm_tn(pooled, self.fc_w, bias=self.fc_b)
        self.static_logits.copy_(logits)

    # -- public ---------------------------------------------------------------------------------------------------------------
    def __call__(self, images_u8: torch.Tensor) -> torch.Tensor:
        """fp32 logits [n, classes] of a uint8 NHWC batch [n, H, W, 3] (n <= batch; a short batch is zero-padded, then sliced)."""
        n = images_u8.shape[0]
        if n > self.batch or tuple(images_u8.shape[1:]) != tuple(self.static_u8.shape[1:]) or images_u8.dtype != torch.uint8:
            raise ValueError(f"expected uint8 [<= {self.batch}, {self.image_size}, {self.image_size}, 3], got "
                             f"{images_u8.dtype} {tuple(images_u8.shape)}")
        self.static_u8[:n].copy_(images_u8, non_blocking=True)
        if n < self.batch:
            self.static_u8[n:].zero_()
        with torch.no_grad():
            if self.graph is not None:
                self.graph.replay()
            else:
                self._forward()
        return self.static_logits[:n].clone()
