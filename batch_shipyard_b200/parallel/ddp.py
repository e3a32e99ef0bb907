"""Fused data-parallel trainer: one CUDA graph per step, one collective kernel per step.

Design (B200-first, replaces what DDP + NCCL + a separate optimizer do in the
baseline recipe):

* every parameter and every gradient is a view into ONE flat bf16 buffer that
  lives in the communicator's symmetric heap, so there is nothing to bucket or
  copy before communication;
* after backward a single kernel does reduce-scatter (multimem.ld_reduce through
  NVSwitch) -> 1/N scale -> SGD-momentum update of the fp32 master shard this
  rank owns -> bf16 all-gather of the new parameters (multimem.st) -> zeroing of
  the local gradient buffer (ZeRO-1 style optimizer-state sharding for free);
* forward + backward + that kernel are captured in one CUDA graph, so a step
  is a single launch from the host;
* the end-to-end path stages uint8 NHWC batches from pinned host memory with a
  double-buffered copy stream and converts them on the GPU.

Reference counterpart: the launcher only wires ``mpirun``/ssh for user
containers (/root/reference/convoy/batch.py:4362-4486); gradient exchange is
whatever the container's framework does.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Callable, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from ..ops import coll as _coll
from ..ops import fused as _fused


def _round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


@dataclass
class FlatLayout:
    total: int
    offsets: dict  # name -> (offset, numel, shape, channels_last)


class FlatParameters:
    """Re-homes a module's parameters/gradients into flat symmetric buffers."""

    def __init__(self, model: nn.Module, comm: _coll.Communicator, dtype=torch.bfloat16):
        self.model, self.comm, self.dtype = model, comm, dtype
        named = [(n, p) for n, p in model.named_parameters() if p.requires_grad]
        off, lay = 0, {}
        for n, p in named:
            lay[n] = (off, p.numel(), tuple(p.shape), p.dim() == 4)
            # every tensor starts on a 256-byte boundary.  Measured (gpurun_out/c5_bench.err, "rerace"): with 16-byte aligned weights
            # the TMA loads of the weight operand (128-byte rows straddling two cache lines) slow the short-K 1x1 GEMMs down by up to
            # 2x (64 -> 64 channels: dgrad 83 us vs 39 us with an aligned weight); cuDNN keeps its weights in registers and does not care.
            off = _round_up(off + p.numel(), 128)
        total = _round_up(off, 8 * max(1, comm.world))
        self.layout = FlatLayout(total, lay)
        dev = comm.torch_device
        # fp32 image of the initial weights (identical on every rank: same seed)
        init = torch.zeros(total, dtype=torch.float32, device=dev)
        for n, p in named:
            o, cnt, shape, cl = lay[n]
            src = p.detach().to(dev, torch.float32)
            if cl:
                src = src.permute(0, 2, 3, 1).contiguous()
            init[o:o + cnt].copy_(src.reshape(-1))
        self.params = comm.alloc(total, dtype)
        self.grads = comm.alloc(total, dtype)
        self.params.copy_(init.to(dtype))
        self.grads.zero_()
        lo, cnt = comm.shard_range(total)
        self.shard = (lo, cnt)
        self.master = init[lo:lo + cnt].clone()
        self.momentum = torch.zeros(cnt, dtype=torch.float32, device=dev)
        del init
        for n, p in named:
            o, cnt_p, shape, cl = lay[n]
            pv, gv = self.params[o:o + cnt_p], self.grads[o:o + cnt_p]
            if cl:
                co, ci, kh, kw = shape
                pv = pv.view(co, kh, kw, ci).permute(0, 3, 1, 2)   # NHWC storage, NCHW logical
                gv = gv.view(co, kh, kw, ci).permute(0, 3, 1, 2)
            else:
                pv, gv = pv.view(shape), gv.view(shape)
            p.data = pv
            p.grad = gv
        for b in model.buffers():
            b.data = b.data.to(dev)

    def checksum(self) -> float:
        return float(self.params.float().sum())


class FusedDataParallelTrainer:
    """Owns the model replica, the flat buffers and the captured training step."""

    def __init__(self, model: nn.Module, comm: _coll.Communicator, batch_shape, num_classes: int,
                 lr: float = 0.1, momentum: float = 0.9, weight_decay: float = 1e-4,
                 loss_fn: Optional[Callable] = None, use_graph: bool = True, channels_last: bool = True):
        self.comm, self.model = comm, model
        self.dev = comm.torch_device
        self.is_cuda = self.dev.type == "cuda"
        if self.is_cuda:
            torch.backends.cudnn.benchmark = True     # the conv dispatcher compares against cuDNN's best algorithm
        self.flat = FlatParameters(model, comm, torch.bfloat16 if self.is_cuda else torch.float32)
        self.hyper = torch.tensor([lr, momentum, weight_decay, 1.0 / comm.world], dtype=torch.float32, device=self.dev)
        self.loss_fn = loss_fn or (lambda logits, y: F.cross_entropy(logits.float(), y))
        n, c, h, w = batch_shape
        self.batch_shape = batch_shape
        act_dtype = torch.bfloat16 if self.is_cuda else torch.float32
        # NHWC storage viewed as NCHW (= torch channels_last).  On CUDA the stem takes a zero-bordered
        # space-to-depth input [N, H/2+3, W/2+3, 16] so its 7x7/s2 conv runs as a dense 4x4 conv.
        self.s2d = bool(self.is_cuda and getattr(model, "s2d_stem", False) and c == 3 and h % 2 == 0 and w % 2 == 0)
        if self.s2d:
            self._x_store = torch.zeros((n, h // 2 + 3, w // 2 + 3, 16), dtype=act_dtype, device=self.dev)
        else:
            self._x_store = torch.zeros((n, h, w, c), dtype=act_dtype, device=self.dev)
        self.static_x = self._x_store.permute(0, 3, 1, 2) if channels_last else self._x_store.permute(0, 3, 1, 2).contiguous()
        self.static_y = torch.zeros((n,), dtype=torch.int64, device=self.dev)
        self.static_loss = torch.zeros((), dtype=torch.float32, device=self.dev)
        self.graph = None
        self.use_graph = use_graph and self.is_cuda
        self.kernels_per_step = 0          # OUR kernels inside one step (graph replays included)
        self.steps_done = 0
        self._stager = None
        model.train()

    # -- one optimisation step on the static buffers ---------------------------
    def _step_body(self) -> None:
        if self.is_cuda:
            _fused.zero_pool_begin(self.dev)            # ONE memset for every layer's zeroed scratch / statistics buffer of this step
        try:
            logits = self.model(self.static_x)
            loss = self.loss_fn(logits, self.static_y)
            loss.backward()
        finally:
            if self.is_cuda:
                _fused.zero_pool_end()
        self.comm.fused_allreduce_sgd(self.flat.grads, self.flat.params, self.flat.master, self.flat.momentum,
                                      self.hyper, zero_grads=True)
        self.static_loss.copy_(loss.detach())

    def _count_own_launches(self) -> int:
        return self.comm.launches + _fused.launch_count() + _extra_launches()

    def prepare(self, warmup: int = 3) -> None:
        """Eager warm-up (also lets cuDNN pick algorithms), then capture the step."""
        # the first eager step autotunes every conv shape (ops.conv) and cuDNN searches its algorithms: ranks can drift apart
        # by seconds, so the collective watchdog is relaxed until the step has been captured
        old_timeout = None
        try:
            old_timeout = self.comm.get_tuning("timeout_ms")
            self.comm.set_tuning(timeout_ms=180000)
        except Exception:  # noqa: BLE001
            old_timeout = None
        def restore():
            if old_timeout:
                self.comm.set_tuning(timeout_ms=int(old_timeout))
        try:
            self._prepare(warmup, restore)
        finally:
            restore()

    def _prepare(self, warmup: int, before_capture=lambda: None) -> None:
        if not self.use_graph:
            before = self._count_own_launches()
            self._step_body()
            self.kernels_per_step = self._count_own_launches() - before
            for _ in range(max(0, warmup - 1)):
                self._step_body()
            return
        s = torch.cuda.Stream(self.dev)
        s.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(s):
            for _ in range(max(1, warmup)):
                self._step_body()
        torch.cuda.current_stream(self.dev).wait_stream(s)
        torch.cuda.synchronize(self.dev)
        before_capture()                       # the captured collective carries the normal watchdog, not the relaxed one
        self.graph = torch.cuda.CUDAGraph()
        before = self._count_own_launches()
        with torch.cuda.graph(self.graph):
            self._step_body()
        self.kernels_per_step = self._count_own_launches() - before
        torch.cuda.synchronize(self.dev)

    def step(self) -> torch.Tensor:
        """Run one step on whatever is in static_x/static_y; returns the loss tensor (device)."""
        if self.graph is not None:
            self.graph.replay()
        else:
            self._step_body()
        self.steps_done += 1
        return self.static_loss

    def load_images_u8(self, images_u8: torch.Tensor, labels: torch.Tensor) -> None:
        """Fill the static step inputs from a device uint8 NHWC batch (used by benches / tests)."""
        if self.s2d:
            _fused.u8_to_s2d_norm(images_u8, self._x_store)
        elif self.is_cuda:
            _fused.u8_to_bf16_norm(images_u8, self._x_store)
        else:
            self._x_store.copy_(images_u8.to(torch.float32) / 255.0)
        self.static_y.copy_(labels)

    def set_lr(self, lr: float) -> None:
        self.hyper[0:1].fill_(lr)

    # -- evaluation --------------------------------------------------------------
    def evaluate(self, images_u8: torch.Tensor, labels: torch.Tensor, batch: Optional[int] = None) -> dict:
        """Held-out metrics of this rank's shard, summed over all ranks: {"count", "loss" (summed cross-entropy), "top1", "top5"}.

        ResNet models on a GPU run on ``parallel.infer.ResNetInference`` (built once per batch size and cached); any other model, and
        every CPU run, uses the module's own eval forward under ``no_grad`` on the input conversion training uses, then restores the
        module's train/eval mode.  No training state changes: flat parameters and gradients, fp32 master, momentum, running
        statistics, the static step inputs and the captured step graph stay as they were, so this may run between steps.
        Every rank must call it (the per-rank sums meet in one all-reduce)."""
        from ..models.resnet import ResNet, ResNetCifar
        n_total = int(images_u8.shape[0])
        bs = int(batch or self.batch_shape[0])
        sums = torch.zeros(4, dtype=torch.float64)
        use_engine = self.is_cuda and isinstance(self.model, (ResNet, ResNetCifar))
        eng = None
        if use_engine and n_total > 0:
            engines = self.__dict__.setdefault("_engines", {})
            eng = engines.get(bs)
            if eng is None:
                from .infer import ResNetInference
                eng = engines[bs] = ResNetInference(self.model, bs, image_size=int(images_u8.shape[1]))
        for i in range(0, n_total, bs):
            x = images_u8[i:i + bs].to(self.dev, non_blocking=True)
            y = labels[i:i + bs].to(self.dev, non_blocking=True)
            logits = eng(x) if eng is not None else self._eval_forward(x)
            logits = logits.float()
            k = min(5, logits.shape[1])
            top = logits.topk(k, dim=1).indices
            hit = top == y.view(-1, 1)
            sums += torch.tensor([float(y.numel()), float(F.cross_entropy(logits, y, reduction="sum")),
                                  float(hit[:, 0].sum()), float(hit.any(dim=1).sum())], dtype=torch.float64)
        buf = self.__dict__.get("_eval_sym")
        if buf is None:
            buf = self._eval_sym = self.comm.alloc(4, torch.float64)       # symmetric: the same code runs on every transport
        buf.copy_(sums.to(buf.device))
        self.comm.all_reduce(buf)
        if self.is_cuda:
            torch.cuda.synchronize(self.dev)
        out = buf.cpu().tolist()
        return {"count": int(round(out[0])), "loss": out[1], "top1": int(round(out[2])), "top5": int(round(out[3]))}

    def _eval_forward(self, images_u8: torch.Tensor) -> torch.Tensor:
        """The module's own eval forward on the conversion training uses (not a hot path)."""
        n, h, w, c = images_u8.shape
        if self.is_cuda:
            if self.s2d:
                xs = torch.empty((n, h // 2 + 3, w // 2 + 3, 16), dtype=torch.bfloat16, device=self.dev)
                _fused.u8_to_s2d_norm(images_u8, xs)
            else:
                xs = torch.empty((n, h, w, c), dtype=torch.bfloat16, device=self.dev)
                _fused.u8_to_bf16_norm(images_u8, xs)
        else:
            xs = images_u8.to(torch.float32) / 255.0
        was_training = self.model.training
        self.model.eval()
        try:
            with torch.no_grad():
                return self.model(xs.permute(0, 3, 1, 2))
        finally:
            self.model.train(was_training)

    # -- end-to-end input path -------------------------------------------------
    def make_stager(self, depth: int = 2) -> "InputStager":
        self._stager = InputStager(self, depth)
        return self._stager


class InputStager:
    """Pinned uint8 NHWC host batches -> device through ``libshipyard_stage`` (native/stage/stage.cpp): every prefetch is a ticket on
    the stager's copy stream (ONE cudaMemcpyAsync straight from the pinned batch, issued only after the step that last read the
    slot has finished — an event dependency, the host never blocks), and the training stream is event-chained behind the ticket
    (``sy_stage_stream_wait``) right before our conversion kernel.  The same mover stages files (task ``input_data``, artefacts)
    file -> pinned arena -> HBM; K12 of SURVEY.md §2E, the data path the reference delegates to blobxfer containers
    (/root/reference/convoy/data.py:567-876, scripts/shipyard_blobxfer.sh)."""

    def __init__(self, tr: FusedDataParallelTrainer, depth: int = 2):
        self.tr, self.depth = tr, depth
        n, c, h, w = tr.batch_shape
        dev = tr.dev
        pin = tr.is_cuda
        self.host_x = [torch.empty((n, h, w, c), dtype=torch.uint8, pin_memory=pin) for _ in range(depth)]
        self.host_y = [torch.empty((n,), dtype=torch.int64, pin_memory=pin) for _ in range(depth)]
        self.dev_x = [torch.empty((n, h, w, c), dtype=torch.uint8, device=dev) for _ in range(depth)]
        self.dev_y = [torch.empty((n,), dtype=torch.int64, device=dev) for _ in range(depth)]
        self.host_loss = [torch.zeros((), dtype=torch.float32, pin_memory=pin) for _ in range(depth)]
        self.h2d_bytes = self.host_x[0].numel() + self.host_y[0].numel() * 8
        self.d2h_bytes = 4
        self.native = None
        self._tickets: list = [None] * depth
        if tr.is_cuda:
            from ..ops.stage import Stager          # no torch fallback on a GPU box: a missing extension must fail loudly
            self.native = Stager(dev.index if dev.index is not None else torch.cuda.current_device(), arena_bytes=8 << 20, concurrency=1)
            self.consumed = [torch.cuda.Event() for _ in range(depth)]
            self.loss_ready = [torch.cuda.Event() for _ in range(depth)]
        self._issued = [False] * depth
        self.transfer_seconds = 0.0
        self.transfers = 0
        self.staging_summary_cached = {"path": "host (cpu)"}

    def fill_synthetic(self, seed: int = 0) -> None:
        g = torch.Generator().manual_seed(seed)
        for hx, hy in zip(self.host_x, self.host_y):
            hx.copy_(torch.randint(0, 256, hx.shape, dtype=torch.uint8, generator=g))
            hy.copy_(torch.randint(0, 1000, hy.shape, dtype=torch.int64, generator=g) % 1000)

    def prefetch(self, slot: int) -> None:
        tr = self.tr
        if not tr.is_cuda:
            self.dev_x[slot].copy_(self.host_x[slot]); self.dev_y[slot].copy_(self.host_y[slot])
            return
        self._reap(slot)
        # the copy may only overwrite the slot once the step that read it is done: an event the copy stream waits for
        wait_ev = self.consumed[slot].cuda_event if self._issued[slot] else 0
        hx, hy = self.host_x[slot], self.host_y[slot]
        self._tickets[slot] = (self.native.submit_pinned(hx.data_ptr(), hx.numel(), self.dev_x[slot].data_ptr(), wait_ev),
                               self.native.submit_pinned(hy.data_ptr(), hy.numel() * 8, self.dev_y[slot].data_ptr(), wait_ev))
        self._issued[slot] = True

    def _reap(self, slot: int) -> None:
        """Release the finished tickets of a slot (their bookkeeping; the device buffers are ours) and account their time."""
        ts = self._tickets[slot]
        if ts is None:
            return
        for t in ts:
            self.native.wait(t)
            self.transfer_seconds += self.native.query(t).transfer_seconds
            self.native.release(t)
        self.transfers += 1
        self._tickets[slot] = None

    def run_step(self, slot: int) -> None:
        """Consume a prefetched slot: convert, train one step, start the loss read-back."""
        tr = self.tr
        if tr.is_cuda:
            cur = torch.cuda.current_stream(tr.dev)
            for t in self._tickets[slot]:
                self.native.stream_wait(t, cur.cuda_stream)         # event-chain the step behind the H2D ticket
            if tr.s2d:
                _fused.u8_to_s2d_norm(self.dev_x[slot], tr._x_store)
            else:
                _fused.u8_to_bf16_norm(self.dev_x[slot], tr._x_store)
            tr.static_y.copy_(self.dev_y[slot], non_blocking=True)
            self.consumed[slot].record(cur)
            tr.step()
            self.host_loss[slot].copy_(tr.static_loss, non_blocking=True)
            self.loss_ready[slot].record(cur)
        else:
            x = self.dev_x[slot].to(torch.float32) / 255.0
            tr._x_store.copy_(x)
            tr.static_y.copy_(self.dev_y[slot])
            tr.step()
            self.host_loss[slot].copy_(tr.static_loss)

    def staging_summary(self) -> dict:
        """What moved the inputs (for the bench record)."""
        if self.native is None:
            return {"path": "host (cpu)"}
        st = self.native.stats()
        return {"path": "libshipyard_stage: pinned -> HBM tickets on the stager's copy stream, step event-chained behind the ticket",
                "tickets": self.transfers * 2, "memcpy_calls": st["memcpy_calls"], "bytes_staged": st["bytes_staged"]}

    def close(self) -> None:
        if self.native is not None:
            for s in range(self.depth):
                self._reap(s)
            self.staging_summary_cached = self.staging_summary()
            self.native.close()
            self.native = None

    def read_loss(self, slot: int) -> float:
        if self.tr.is_cuda:
            self.loss_ready[slot].synchronize()
        return float(self.host_loss[slot])


_EXTRA_COUNTERS: list = []


def register_launch_counter(fn: Callable[[], int]) -> None:
    """Other native op libraries (GEMM, ...) register their launch counters here."""
    _EXTRA_COUNTERS.append(fn)


def _extra_launches() -> int:
    return sum(int(f()) for f in _EXTRA_COUNTERS)
