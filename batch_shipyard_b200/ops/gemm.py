"""ctypes binding + autograd wrappers for ``libshipyard_gemm`` (tcgen05/TMEM/TMA bf16 GEMM and implicit-GEMM convolution).

The reference ships no compute kernels (its GPU recipes launch framework containers, e.g.
/root/reference/recipes/PyTorch-GPU/config/jobs.yaml:1-8 and /root/reference/recipes/CNTK-GPU-OpenMPI/docker/run_cntk.sh:66-78);
these are the tensor-core half of the retargeted recipes (SURVEY.md §2E rows K10, K12).

``gemm_tn(a, b)`` computes ``a @ b.T`` for row-major bf16 ``a[M,K]``, ``b[N,K]`` — the shape of a
``Linear`` and of a 1x1 convolution on NHWC activations (``X[M=N*H*W, Cin] @ W[Cout, Cin]^T``).
With ``stats=`` the kernel's epilogue also accumulates the per-channel sum and sum of squares
of the output, i.e. the train-mode BatchNorm statistics, saving one full pass over the activations.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_LIB = None


def lib_path() -> str:
    return os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "_native", "libshipyard_gemm.so")


def load() -> C.CDLL:
    global _LIB
    if _LIB is None:
        p = lib_path()
        if not os.path.exists(p):
            from .._build import ensure_built
            ensure_built(["gemm"])
        if not os.path.exists(p):
            raise RuntimeError(f"{p} missing: run `python native/build.py gemm` (no fallback on GPU)")
        lib = C.CDLL(p)
        lib.sy_gemm_last_error.restype = C.c_char_p
        lib.sy_gemm_launch_count.restype = C.c_ulonglong
        lib.sy_gemm_bf16_tn.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                        C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        lib.sy_gemm_bf16_tn_allreduce.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_int,
                                                  C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
        lib.sy_gemm_bf16_nn.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                        C.c_int, C.c_int, C.c_void_p]
        lib.sy_gemm_bf16_nt_splitk.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                               C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]
        lib.sy_gemm_bf16_tn_rsag.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int,
                                             C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.c_void_p]
        lib.sy_gemm_bf16_tn_2cta.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int] * 6 + [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]
        lib.sy_conv_bf16_nhwc_2cta.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int] * 10 + [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        lib.sy_conv_bf16_wgrad.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int] * 9 + [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]
        lib.sy_conv_bf16_nhwc.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int] * 10 + [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        lib.sy_conv3x3_halo.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int] * 6 + [C.c_void_p] + [C.c_int] * 4 + [C.c_void_p]
        lib.sy_conv3x3_halo_rows.argtypes = [C.c_int, C.c_int]
        lib.sy_conv3x3_wgrad_halo.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int] * 5 + [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        lib.sy_gemm_bf16_nn_scatter2.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int] * 7 + [C.c_void_p]
        lib.sy_stem_s2d_fprop.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
        lib.sy_gemm_bf16_tn_affine.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int] * 6 + [C.c_void_p, C.c_void_p, C.c_void_p] + \
            [C.c_int] * 4 + [C.c_void_p]
        lib.sy_conv_bf16_nhwc_affine.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int] * 9 + [C.c_void_p, C.c_void_p, C.c_void_p] + \
            [C.c_int] * 3 + [C.c_void_p]
        lib.sy_stem_s2d_wgrad.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                          C.c_void_p]
        _LIB = lib
        try:
            from ..parallel.ddp import register_launch_counter
            register_launch_counter(lambda: int(lib.sy_gemm_launch_count()))
        except Exception:  # noqa: BLE001
            pass
    return _LIB


def _pool_zeros(n: int, device) -> torch.Tensor:
    from .fused import zeros            # slice of the training step's zero pool when one is open, else torch.zeros
    return zeros(n, device)


def launch_count() -> int:
    return int(load().sy_gemm_launch_count())


def _rows_ok(t: torch.Tensor) -> bool:
    return t.dim() == 2 and t.stride(1) == 1 and t.stride(0) % 8 == 0 and t.data_ptr() % 16 == 0


def two_cta_ok(m: int, n: int, block_n: int = 0) -> bool:
    """Shapes the CTA-pair (cta_group::2, M = 256) kernels accept."""
    bn = block_n or (256 if n % 256 == 0 else 128)
    return n % bn == 0 and bn in (128, 256)


def gemm_tn(a: torch.Tensor, b: torch.Tensor, out: Optional[torch.Tensor] = None, bias: Optional[torch.Tensor] = None,
            stats: Optional[torch.Tensor] = None, block_n: int = 0, max_ctas: int = 0, two_cta: bool = False) -> torch.Tensor:
    """out[M,N] = a[M,K] @ b[N,K]^T (+ bias[N]); bf16, fp32 accumulation in TMEM.
    stats: zero-initialised float32[2*N] receiving column sums / sums of squares of `out`."""
    assert a.is_cuda and a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16 and a.shape[1] == b.shape[1]
    m, k = a.shape
    n = b.shape[0]
    if k % 8:                                   # TMA needs 16-byte row pitches: zero-pad K (zeros do not change the product)
        pad = 8 - k % 8
        a = torch.nn.functional.pad(a, (0, pad)); b = torch.nn.functional.pad(b, (0, pad)); k += pad
    if not _rows_ok(a):
        a = a.contiguous()
    if not _rows_ok(b):
        b = b.contiguous()
    if out is None:
        ldc = (n + 7) // 8 * 8
        buf = torch.empty((m, ldc), dtype=torch.bfloat16, device=a.device)
        out = buf[:, :n] if ldc != n else buf
    assert out.shape == (m, n) and out.dtype == torch.bfloat16 and _rows_ok(out)
    if stats is not None:
        assert stats.dtype == torch.float32 and stats.numel() == 2 * n and stats.is_contiguous()
    if bias is not None:
        assert bias.dtype == torch.bfloat16 and bias.numel() == n and bias.is_contiguous()
    lib = load()
    if two_cta:
        assert bias is None and two_cta_ok(m, n, block_n), "2-CTA GEMM: no bias, N % block_n == 0"
        rc = lib.sy_gemm_bf16_tn_2cta(C.c_void_p(a.data_ptr()), C.c_void_p(b.data_ptr()), C.c_void_p(out.data_ptr()), m, n, k,
                                      a.stride(0), b.stride(0), out.stride(0), C.c_void_p(stats.data_ptr() if stats is not None else 0),
                                      block_n, max_ctas, 0, C.c_void_p(torch.cuda.current_stream(a.device).cuda_stream))
        if rc != 0:
            raise RuntimeError(f"sy_gemm_bf16_tn_2cta failed ({rc}): {lib.sy_gemm_last_error().decode()}")
        return out
    rc = lib.sy_gemm_bf16_tn(C.c_void_p(a.data_ptr()), C.c_void_p(b.data_ptr()), C.c_void_p(out.data_ptr()), m, n, k,
                             a.stride(0), b.stride(0), out.stride(0), C.c_void_p(bias.data_ptr() if bias is not None else 0),
                             C.c_void_p(stats.data_ptr() if stats is not None else 0), block_n, max_ctas,
                             C.c_void_p(torch.cuda.current_stream(a.device).cuda_stream))
    if rc != 0:
        raise RuntimeError(f"sy_gemm_bf16_tn failed ({rc}): {lib.sy_gemm_last_error().decode()}")
    return out


def gemm_nn(a: torch.Tensor, b: torch.Tensor, out: Optional[torch.Tensor] = None, block_n: int = 0, max_ctas: int = 0,
            two_cta: bool = False) -> torch.Tensor:
    """out[M,N] = a[M,K] @ b[K,N] with b row-major (N contiguous): the dgrad shape dX = dY @ W.  The kernel reads b as an
    MN-major tcgen05 operand, so no transposed copy of the weight is made."""
    assert a.is_cuda and a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16 and a.shape[1] == b.shape[0]
    m, k = a.shape
    n = b.shape[1]
    if not _rows_ok(a):
        a = a.contiguous()
    if not _rows_ok(b):
        b = b.contiguous()
    if k % 8 or not _rows_ok(a):
        return gemm_tn(a, b.t().contiguous(), out=out, block_n=block_n, max_ctas=max_ctas)
    if out is None:
        ldc = (n + 7) // 8 * 8
        buf = torch.empty((m, ldc), dtype=torch.bfloat16, device=a.device)
        out = buf[:, :n] if ldc != n else buf
    assert out.shape == (m, n) and out.dtype == torch.bfloat16 and _rows_ok(out)
    lib = load()
    if two_cta:
        assert two_cta_ok(m, n, block_n), "2-CTA GEMM: N % block_n == 0"
        rc = lib.sy_gemm_bf16_tn_2cta(C.c_void_p(a.data_ptr()), C.c_void_p(b.data_ptr()), C.c_void_p(out.data_ptr()), m, n, k,
                                      a.stride(0), b.stride(0), out.stride(0), None, block_n, max_ctas, 1,
                                      C.c_void_p(torch.cuda.current_stream(a.device).cuda_stream))
        if rc != 0:
            raise RuntimeError(f"sy_gemm_bf16_tn_2cta (MN-major B) failed ({rc}): {lib.sy_gemm_last_error().decode()}")
        return out
    rc = lib.sy_gemm_bf16_nn(C.c_void_p(a.data_ptr()), C.c_void_p(b.data_ptr()), C.c_void_p(out.data_ptr()), m, n, k,
                             a.stride(0), b.stride(0), out.stride(0), block_n, max_ctas,
                             C.c_void_p(torch.cuda.current_stream(a.device).cuda_stream))
    if rc != 0:
        raise RuntimeError(f"sy_gemm_bf16_nn failed ({rc}): {lib.sy_gemm_last_error().decode()}")
    return out


_WS: dict = {}
_WS_FLOATS = 4 << 20          # covers I*J up to 2048 x 2048
_WS_TICKETS = 4096


def _workspace(dev: torch.device):
    """Per-device split-K workspace: zero on entry AND on exit of every wgrad kernel (the finalising CTA cleans up),
    so one allocation serves every layer and the kernel stays CUDA-graph capturable."""
    key = (dev.type, dev.index)
    if key not in _WS:
        _WS[key] = (torch.zeros(_WS_FLOATS, dtype=torch.float32, device=dev), torch.zeros(_WS_TICKETS, dtype=torch.int32, device=dev))
    return _WS[key]


def conv1x1_s2_dgrad(dy: torch.Tensor, w: torch.Tensor, block_n: int = 0, max_ctas: int = 0) -> torch.Tensor:
    """dX[N, Cin, 2P, 2Q] of a 1x1 / stride-2 convolution (the ResNet downsample branches) from dY[N, Cout, P, Q] (channels_last) and
    W[Cout, Cin, 1, 1]: ONE tcgen05 GEMM (weights read in place as an MN-major operand) whose st.global epilogue scatters row (n, p, q)
    to pixel (2p, 2q) and writes the zeros of the three pixels the forward pass skipped — no memset, no strided copy."""
    n, cout, p, q = dy.shape
    cin = w.shape[1]
    dys, ws_ = _nhwc_storage(dy), _nhwc_storage(w)
    dx = torch.empty((n, 2 * p, 2 * q, cin), dtype=torch.bfloat16, device=dy.device)
    lib = load()
    rc = lib.sy_gemm_bf16_nn_scatter2(C.c_void_p(dys.data_ptr()), C.c_void_p(ws_.data_ptr()), C.c_void_p(dx.data_ptr()), n, p, q, cout, cin,
                                      block_n, max_ctas, C.c_void_p(torch.cuda.current_stream(dy.device).cuda_stream))
    if rc != 0:
        raise RuntimeError(f"sy_gemm_bf16_nn_scatter2 failed ({rc}): {lib.sy_gemm_last_error().decode()}")
    return dx.permute(0, 3, 1, 2)


def gemm_nt_wgrad(a: torch.Tensor, b: torch.Tensor, out: Optional[torch.Tensor] = None, accumulate: bool = False,
                  block_n: int = 0, splits: int = 0) -> torch.Tensor:
    """out[J, I] (+)= b[K,J]^T @ a[K,I]  — the weight gradient dW[Cout,Cin] = dY^T X with a = X[pixels,Cin], b = dY[pixels,Cout].
    One split-K tcgen05 kernel (both operands MN-major through TMA); the last CTA of a tile writes bf16 into `out`."""
    assert a.is_cuda and a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16 and a.shape[0] == b.shape[0]
    k, i = a.shape
    j = b.shape[1]
    if not _rows_ok(a):
        a = a.contiguous()
    if not _rows_ok(b):
        b = b.contiguous()
    assert _rows_ok(a) and _rows_ok(b), "wgrad operands need 16-byte aligned rows (channel counts multiple of 8)"
    if out is None:
        out = torch.empty((j, i), dtype=torch.bfloat16, device=a.device)
        accumulate = False
    assert out.shape == (j, i) and out.dtype == torch.bfloat16 and out.stride(1) == 1
    ws, tickets = _workspace(a.device)
    if i * j > ws.numel():
        raise RuntimeError(f"wgrad output {j}x{i} exceeds the split-K workspace")
    lib = load()
    rc = lib.sy_gemm_bf16_nt_splitk(C.c_void_p(a.data_ptr()), C.c_void_p(b.data_ptr()), C.c_void_p(out.data_ptr()), i, j, k,
                                    a.stride(0), b.stride(0), out.stride(0), C.c_void_p(ws.data_ptr()), C.c_void_p(tickets.data_ptr()),
                                    1 if accumulate else 0, block_n, splits, C.c_void_p(torch.cuda.current_stream(a.device).cuda_stream))
    if rc != 0:
        raise RuntimeError(f"sy_gemm_bf16_nt_splitk failed ({rc}): {lib.sy_gemm_last_error().decode()}")
    return out


def _grad_view_2d(p: torch.Tensor, rows: int, cols: int) -> Optional[torch.Tensor]:
    """The parameter's existing .grad as a contiguous [rows, cols] view (NHWC-stored conv weights included), or None."""
    g = getattr(p, "grad", None)
    if g is None or g.dtype != torch.bfloat16:
        return None
    v = g.permute(0, 2, 3, 1) if g.dim() == 4 else g
    if not v.is_contiguous():
        return None
    return v.reshape(rows, cols)


class _LinearTN(torch.autograd.Function):
    """y = x @ w^T (+ b): forward, dgrad (W read as an MN-major operand) and wgrad (split-K, both MN-major) all on tcgen05."""

    @staticmethod
    def forward(ctx, x, w, b):
        ctx.save_for_backward(x, w)
        ctx.has_bias = b is not None
        ctx.w_ref = w
        return gemm_tn(x, w, bias=b)

    @staticmethod
    def backward(ctx, dy):
        x, w = ctx.saved_tensors
        if not _rows_ok(dy):
            dy = dy.contiguous()
        dx = gemm_nn(dy, w) if ctx.needs_input_grad[0] else None                        # dX = dY @ W
        dw = None
        if ctx.needs_input_grad[1]:
            gv = _grad_view_2d(ctx.w_ref, w.shape[0], w.shape[1])
            if gv is not None and x.shape[1] % 8 == 0 and _rows_ok(dy):
                gemm_nt_wgrad(x, dy, out=gv, accumulate=True)                           # straight into the flat gradient buffer
            elif x.shape[1] % 8 == 0 and _rows_ok(dy):
                dw = gemm_nt_wgrad(x, dy)
            else:
                dw = dy.t() @ x
        db = dy.float().sum(0).to(dy.dtype) if ctx.has_bias else None
        return dx, dw, db


def linear(x: torch.Tensor, w: torch.Tensor, b: Optional[torch.Tensor] = None) -> torch.Tensor:
    return _LinearTN.apply(x, w, b)


class _Conv1x1NHWC(torch.autograd.Function):
    """1x1 stride-1 convolution on channels_last bf16 activations as one GEMM; the epilogue produces the
    BatchNorm statistics of the output (returned as a non-differentiable float32[2*Cout])."""

    @staticmethod
    def forward(ctx, x, w, want_stats):
        ctx.set_materialize_grads(False)          # the statistics output has no gradient: do not let autograd build a zeros tensor for it
        n, cin, h, wd = x.shape
        cout = w.shape[0]
        x2 = x.permute(0, 2, 3, 1).reshape(n * h * wd, cin)            # view: NHWC storage
        w2 = w.permute(0, 2, 3, 1).reshape(cout, cin)
        stats = _pool_zeros(2 * cout, x.device) if want_stats else None
        y2 = gemm_tn(x2, w2, stats=stats)
        ctx.save_for_backward(x, w)
        ctx.w_ref = w
        y = y2.view(n, h, wd, cout).permute(0, 3, 1, 2)
        ctx.mark_non_differentiable(stats) if stats is not None else None
        return (y, stats) if want_stats else (y, None)

    @staticmethod
    def backward(ctx, dy, _dstats):
        x, w = ctx.saved_tensors
        n, cin, h, wd = x.shape
        cout = w.shape[0]
        dy2 = dy.permute(0, 2, 3, 1).reshape(n * h * wd, cout)
        if not _rows_ok(dy2):
            dy2 = dy2.contiguous()
        dx = dw = None
        if ctx.needs_input_grad[0]:
            w2 = w.permute(0, 2, 3, 1).reshape(cout, cin)                            # [K=Cout, N=Cin]: MN-major B, no transpose
            dx = gemm_nn(dy2, w2).view(n, h, wd, cin).permute(0, 3, 1, 2)
        if ctx.needs_input_grad[1]:
            x2 = x.permute(0, 2, 3, 1).reshape(n * h * wd, cin)
            gv = _grad_view_2d(ctx.w_ref, cout, cin)
            if gv is not None:
                gemm_nt_wgrad(x2, dy2, out=gv, accumulate=True)                      # written into w.grad by the kernel itself
            else:
                dw = gemm_nt_wgrad(x2, dy2).view(cout, 1, 1, cin).permute(0, 3, 1, 2)
        return dx, dw, None


def conv1x1_nhwc(x: torch.Tensor, w: torch.Tensor, want_stats: bool = False):
    return _Conv1x1NHWC.apply(x, w, want_stats)


def gemm_tn_allreduce(comm, a: torch.Tensor, b: torch.Tensor, out_sym: torch.Tensor, block_n: int = 0) -> torch.Tensor:
    """K10: ``out_sym += a @ b.T`` summed over all ranks, ONE kernel (tcgen05 GEMM whose epilogue issues
    multimem.red into the NVLS multicast mapping of ``out_sym``; ends with a cross-GPU flag barrier).
    ``out_sym``: fp32 [M, N] from ``comm.alloc`` and zero on every rank before the call; a/b: this rank's K-shard."""
    assert a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16 and out_sym.dtype == torch.float32
    m, k = a.shape
    n = b.shape[0]
    assert tuple(out_sym.shape) == (m, n) and out_sym.is_contiguous() and _rows_ok(a) and _rows_ok(b)
    lib = load()
    from . import coll as _coll
    clib = _coll.load()
    clib.sy_comm_device_view.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    clib.sy_comm_device_view.restype = C.c_size_t
    size = clib.sy_comm_device_view(comm._h, None, 0)
    view = (C.c_uint8 * size)()
    clib.sy_comm_device_view(comm._h, view, size)
    rc = lib.sy_gemm_bf16_tn_allreduce(view, size, C.c_void_p(a.data_ptr()), C.c_void_p(b.data_ptr()), comm.heap_offset(out_sym), m, n, k,
                                       a.stride(0), b.stride(0), out_sym.stride(0), block_n,
                                       C.c_void_p(torch.cuda.current_stream(a.device).cuda_stream))
    if rc != 0:
        raise RuntimeError(f"sy_gemm_bf16_tn_allreduce failed ({rc}): {lib.sy_gemm_last_error().decode()}")
    return out_sym


def _comm_view(comm):
    from . import coll as _coll
    clib = _coll.load()
    clib.sy_comm_device_view.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    clib.sy_comm_device_view.restype = C.c_size_t
    size = clib.sy_comm_device_view(comm._h, None, 0)
    view = (C.c_uint8 * size)()
    clib.sy_comm_device_view(comm._h, view, size)
    return view, size


def gemm_tn_allreduce_bf16(comm, a: torch.Tensor, b: torch.Tensor, out_sym: torch.Tensor, inbox: Optional[torch.Tensor] = None,
                           block_n: int = 0) -> torch.Tensor:
    """K10 v2: ``out_sym = sum_ranks(a_r @ b_r.T)`` in ONE kernel with a reduce-scatter / all-gather schedule and bf16 on
    the wire: partial tiles are stored straight from TMEM into the owning rank's inbox over NVLink, the owner reduces in
    fp32 and multicasts the bf16 result (multimem.st).  ``out_sym``: bf16 [M, N] from ``comm.alloc`` (no zeroing needed)."""
    assert a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16 and out_sym.dtype == torch.bfloat16
    m, k = a.shape
    n = b.shape[0]
    assert tuple(out_sym.shape) == (m, n) and out_sym.is_contiguous() and _rows_ok(a) and _rows_ok(b) and n % 8 == 0
    lib = load()
    view, size = _comm_view(comm)
    rpr = C.c_int(0)
    lib.sy_gemm_bf16_tn_rsag(view, size, None, None, 0, 0, m, n, k, 8, 8, block_n, C.byref(rpr), None)
    need = comm.world * rpr.value * n
    if inbox is None:
        cache = comm.__dict__.setdefault("_k10_inbox", {})
        inbox = cache.get(need)
        if inbox is None:
            inbox = cache[need] = comm.alloc(need, torch.bfloat16)
    assert inbox.dtype == torch.bfloat16 and inbox.numel() >= need
    rc = lib.sy_gemm_bf16_tn_rsag(view, size, C.c_void_p(a.data_ptr()), C.c_void_p(b.data_ptr()), comm.heap_offset(inbox),
                                  comm.heap_offset(out_sym), m, n, k, a.stride(0), b.stride(0), block_n, C.byref(rpr),
                                  C.c_void_p(torch.cuda.current_stream(a.device).cuda_stream))
    if rc != 0:
        raise RuntimeError(f"sy_gemm_bf16_tn_rsag failed ({rc}): {lib.sy_gemm_last_error().decode()}")
    return out_sym


# ---------------------------------------------------------------------------------------------------------
# Convolution as implicit GEMM (TMA im2col loads feeding tcgen05; no im2col buffer)
# ---------------------------------------------------------------------------------------------------------
def _nhwc_storage(t: torch.Tensor) -> torch.Tensor:
    """[N,C,H,W] channels_last tensor -> its dense [N,H,W,C] storage view (copy only if it is not channels_last)."""
    v = t.permute(0, 2, 3, 1)
    return v if v.is_contiguous() else v.contiguous()


def conv_supported(x: torch.Tensor, w: torch.Tensor, stride: int, pad: int) -> bool:
    n, cin, h, wd = x.shape
    cout, _, r, s = w.shape
    p, q = (h + 2 * pad - r) // stride + 1, (wd + 2 * pad - s) // stride + 1
    return (x.is_cuda and x.dtype == torch.bfloat16 and cin % 64 == 0 and cout % 8 == 0 and (n * p * q) % 128 == 0)


def conv_fprop_nhwc(x: torch.Tensor, w: torch.Tensor, stride: int = 1, pad: int = 1, stats: Optional[torch.Tensor] = None,
                    block_n: int = 0, max_ctas: int = 0, two_cta: bool = False) -> torch.Tensor:
    """y = conv2d(x, w) for channels_last bf16 x[N,Cin,H,W], w[Cout,Cin,R,S] (stored KRSC); returns channels_last y."""
    n, cin, h, wd = x.shape
    cout, _, r, s = w.shape
    p, q = (h + 2 * pad - r) // stride + 1, (wd + 2 * pad - s) // stride + 1
    xs, ws = _nhwc_storage(x), _nhwc_storage(w)
    y = torch.empty((n, p, q, cout), dtype=torch.bfloat16, device=x.device)
    lib = load()
    if two_cta:
        rc = lib.sy_conv_bf16_nhwc_2cta(C.c_void_p(xs.data_ptr()), C.c_void_p(ws.data_ptr()), C.c_void_p(y.data_ptr()), n, h, wd, cin, cout, r, s,
                                        pad, stride, 0, C.c_void_p(stats.data_ptr() if stats is not None else 0), block_n, max_ctas,
                                        C.c_void_p(torch.cuda.current_stream(x.device).cuda_stream))
        if rc != 0:
            raise RuntimeError(f"sy_conv_bf16_nhwc_2cta failed ({rc}): {lib.sy_gemm_last_error().decode()}")
        return y.permute(0, 3, 1, 2)
    rc = lib.sy_conv_bf16_nhwc(C.c_void_p(xs.data_ptr()), C.c_void_p(ws.data_ptr()), C.c_void_p(y.data_ptr()), n, h, wd, cin, cout, r, s,
                               pad, stride, 0, C.c_void_p(stats.data_ptr() if stats is not None else 0), block_n, max_ctas,
                               C.c_void_p(torch.cuda.current_stream(x.device).cuda_stream))
    if rc != 0:
        raise RuntimeError(f"sy_conv_bf16_nhwc fprop failed ({rc}): {lib.sy_gemm_last_error().decode()}")
    return y.permute(0, 3, 1, 2)


def halo_rows(h: int, w: int) -> int:
    """Image rows per M tile of the halo-load 3x3 kernel: the largest divisor R of H with R*(W+2) <= 128 (0 = unsupported).
    Pure-Python mirror of ``halo_rows`` in native/gemm/conv_halo.inc so the dispatcher can filter shapes without a GPU."""
    wp, best = w + 2, 0
    for r in range(1, h + 1):
        if h % r == 0 and r * wp <= 128 and (r + 2) * wp <= 256 and wp <= 256:
            best = r
    return best


def halo_ok(n: int, h: int, w: int, c_act: int, c_out: int, r: int, s: int, stride: int, pad: int, pair: bool = False,
            dgrad: bool = False) -> bool:
    """Shapes the halo-load kernel accepts: 3x3, stride 1, pad 1, activation channels % 64, whole image rows per tile."""
    if (r, s, stride, pad) != (3, 3, 1, 1) or c_act % 64 or c_out % (64 if dgrad else 8):
        return False
    rows = halo_rows(h, w)
    if rows == 0:
        return False
    if pair:
        return c_out % 128 == 0 and (n * (h // rows)) % 2 == 0
    return True


# A-descriptor base_offset for the row-shifted taps: 0.  Measured on B200 (profiles/conv_halo.md): tcgen05 applies the 128-byte
# swizzle to the absolute shared-memory address, so a start address that is not 1024-byte aligned needs NO base offset when the
# data was written by TMA into a 1024-byte aligned buffer; setting base_offset = (addr >> 7) & 7 gives wrong results.
_HALO_BASE_MODE = int(os.environ.get("SHIPYARD_HALO_BASE_MODE", "0"))


def conv3x3_halo(act: torch.Tensor, w: torch.Tensor, dgrad: bool = False, stats: Optional[torch.Tensor] = None, block_n: int = 0,
                 pair: bool = False, base_mode: Optional[int] = None, max_ctas: int = 0, epi_alt: bool = False,
                 weights_stationary: bool = False) -> torch.Tensor:
    """3x3 / stride 1 / pad 1 convolution through the halo-load kernel (native/gemm/conv_halo.inc).

    fprop: ``act`` = x[N,Cin,H,W], ``w`` = W[Cout,Cin,3,3] -> y[N,Cout,H,W] (optionally the BN statistics of y in ``stats``);
    dgrad: ``act`` = dY[N,Cout,H,W], same ``w`` -> dX[N,Cin,H,W].  channels_last bf16 in and out.

    ``epi_alt`` (64 output channels, no pair: the two epilogue warpgroups take alternate tiles) and ``weights_stationary``
    (pair, 128 output channels, 128 input channels, 28x28-class images: all 18 weight tiles stay in shared memory) select
    variants written after the last GPU run of round 1 — compiled, reviewed, not yet validated on hardware; off by default."""
    n, ca, h, wd = act.shape
    cn = w.shape[1] if dgrad else w.shape[0]
    a_s, w_s = _nhwc_storage(act), _nhwc_storage(w)
    y = torch.empty((n, h, wd, cn), dtype=torch.bfloat16, device=act.device)
    lib = load()
    rc = lib.sy_conv3x3_halo(C.c_void_p(a_s.data_ptr()), C.c_void_p(w_s.data_ptr()), C.c_void_p(y.data_ptr()), n, h, wd, ca, cn,
                             1 if dgrad else 0, C.c_void_p(stats.data_ptr() if stats is not None else 0), block_n, 1 if pair else 0,
                             (_HALO_BASE_MODE if base_mode is None else base_mode) | (2 if epi_alt else 0) | (4 if weights_stationary else 0),
                             max_ctas,
                             C.c_void_p(torch.cuda.current_stream(act.device).cuda_stream))
    if rc != 0:
        raise RuntimeError(f"sy_conv3x3_halo failed ({rc}): {lib.sy_gemm_last_error().decode()}")
    return y.permute(0, 3, 1, 2)


def conv3x3_wgrad_halo(x: torch.Tensor, dy: torch.Tensor, out: Optional[torch.Tensor] = None, accumulate: bool = False,
                       splits: int = 0) -> torch.Tensor:
    """dW[Cout,Cin,3,3] (stored KRSC) of a 3x3 / stride-1 / pad-1 convolution through the halo-load wgrad kernel
    (native/gemm/wgrad_halo.inc): X and dY are read once per (64 ci, 64 co) block, the nine taps are row-shifted descriptors of one
    X halo box.  NOT yet validated on hardware (written after the last GPU run of round 1); nothing selects it by default."""
    n, cin, h, wd = x.shape
    cout = dy.shape[1]
    xs, dys = _nhwc_storage(x), _nhwc_storage(dy)
    if out is None:
        out = torch.empty((cout, 3, 3, cin), dtype=torch.bfloat16, device=x.device)
        accumulate = False
    assert out.is_contiguous() and tuple(out.shape) == (cout, 3, 3, cin) and out.dtype == torch.bfloat16
    ws, tickets = _workspace(x.device)
    if 9 * cin * cout > ws.numel() or (cin // 64) * (cout // 64) > tickets.numel():
        raise RuntimeError("conv wgrad output exceeds the split-K workspace")
    lib = load()
    rc = lib.sy_conv3x3_wgrad_halo(C.c_void_p(xs.data_ptr()), C.c_void_p(dys.data_ptr()), C.c_void_p(out.data_ptr()), n, h, wd, cin, cout,
                                   C.c_void_p(ws.data_ptr()), C.c_void_p(tickets.data_ptr()), 1 if accumulate else 0, splits,
                                   C.c_void_p(torch.cuda.current_stream(x.device).cuda_stream))
    if rc != 0:
        raise RuntimeError(f"sy_conv3x3_wgrad_halo failed ({rc}): {lib.sy_gemm_last_error().decode()}")
    return out.permute(0, 3, 1, 2)


def conv_two_cta_ok(n: int, p: int, q: int, c_out: int) -> bool:
    return (n * p * q) % 256 == 0 and c_out % 128 == 0


def conv_dgrad_nhwc(dy: torch.Tensor, w: torch.Tensor, pad: int = 1, block_n: int = 0, two_cta: bool = False) -> torch.Tensor:
    """dx of a stride-1 'same' convolution: implicit GEMM over dY with the weights read in place (rotated by tap index,
    transposed by reading them as an MN-major operand)."""
    n, cout, p, q = dy.shape
    _, cin, r, s = w.shape
    dys, ws = _nhwc_storage(dy), _nhwc_storage(w)
    dx = torch.empty((n, p, q, cin), dtype=torch.bfloat16, device=dy.device)
    lib = load()
    if two_cta:
        rc = lib.sy_conv_bf16_nhwc_2cta(C.c_void_p(dys.data_ptr()), C.c_void_p(ws.data_ptr()), C.c_void_p(dx.data_ptr()), n, p, q, cout, cin, r, s,
                                        pad, 1, 1, None, block_n, 0, C.c_void_p(torch.cuda.current_stream(dy.device).cuda_stream))
        if rc != 0:
            raise RuntimeError(f"sy_conv_bf16_nhwc_2cta dgrad failed ({rc}): {lib.sy_gemm_last_error().decode()}")
        return dx.permute(0, 3, 1, 2)
    rc = lib.sy_conv_bf16_nhwc(C.c_void_p(dys.data_ptr()), C.c_void_p(ws.data_ptr()), C.c_void_p(dx.data_ptr()), n, p, q, cout, cin, r, s,
                               pad, 1, 1, None, block_n, 0, C.c_void_p(torch.cuda.current_stream(dy.device).cuda_stream))
    if rc != 0:
        raise RuntimeError(f"sy_conv_bf16_nhwc dgrad failed ({rc}): {lib.sy_gemm_last_error().decode()}")
    return dx.permute(0, 3, 1, 2)


def conv_wgrad_nhwc(x: torch.Tensor, dy: torch.Tensor, wshape, stride: int = 1, pad: int = 1, out: Optional[torch.Tensor] = None,
                    accumulate: bool = False, block_n: int = 0, splits: int = 0) -> torch.Tensor:
    """dW[Cout,Cin,R,S] (stored KRSC) of conv2d(x, w): one split-K tcgen05 launch over all filter taps, im2col(x) through TMA,
    dY read as an MN-major operand; with `out` (a KRSC-dense [Cout,R,S,Cin] view, e.g. the flat gradient buffer) the last CTA
    of every tile writes / accumulates the bf16 gradient in place."""
    n, cin, h, wd = x.shape
    cout, _, r, s = wshape
    xs, dys = _nhwc_storage(x), _nhwc_storage(dy)
    if out is None:
        out = torch.empty((cout, r, s, cin), dtype=torch.bfloat16, device=x.device)
        accumulate = False
    assert out.is_contiguous() and tuple(out.shape) == (cout, r, s, cin) and out.dtype == torch.bfloat16
    ws, tickets = _workspace(x.device)
    if r * s * cin * cout > ws.numel():
        raise RuntimeError("conv wgrad output exceeds the split-K workspace")
    lib = load()
    rc = lib.sy_conv_bf16_wgrad(C.c_void_p(xs.data_ptr()), C.c_void_p(dys.data_ptr()), C.c_void_p(out.data_ptr()), n, h, wd, cin, cout, r, s,
                                pad, stride, C.c_void_p(ws.data_ptr()), C.c_void_p(tickets.data_ptr()), 1 if accumulate else 0, block_n, splits,
                                C.c_void_p(torch.cuda.current_stream(x.device).cuda_stream))
    if rc != 0:
        raise RuntimeError(f"sy_conv_bf16_wgrad failed ({rc}): {lib.sy_gemm_last_error().decode()}")
    return out.permute(0, 3, 1, 2)


class _ConvNHWC(torch.autograd.Function):
    """KxK (strided) convolution on channels_last bf16 activations, all three passes on tcgen05 implicit-GEMM kernels:
    fprop (+ BN statistics), stride-1 dgrad (weights read in place), wgrad (split-K over pixels, all taps in one launch)."""

    @staticmethod
    def forward(ctx, x, w, stride, pad, want_stats):
        ctx.set_materialize_grads(False)          # the statistics output has no gradient: do not let autograd build a zeros tensor for it
        cout = w.shape[0]
        stats = _pool_zeros(2 * cout, x.device) if want_stats else None
        y = conv_fprop_nhwc(x, w, stride, pad, stats=stats)
        ctx.save_for_backward(x, w)
        ctx.stride, ctx.pad = stride, pad
        ctx.w_ref = w
        if stats is not None:
            ctx.mark_non_differentiable(stats)
        return y, stats

    @staticmethod
    def backward(ctx, dy, _ds):
        x, w = ctx.saved_tensors
        dx = dw = None
        if not dy.is_contiguous(memory_format=torch.channels_last):
            dy = dy.contiguous(memory_format=torch.channels_last)
        if ctx.needs_input_grad[0]:
            if ctx.stride == 1 and dy.shape[1] % 64 == 0 and dy.shape[2:] == x.shape[2:]:
                dx = conv_dgrad_nhwc(dy, w, ctx.pad)
            else:                        # strided dgrad: cuDNN on the channels_last tensors (no layout round trip)
                dx = torch.ops.aten.convolution_backward(dy, x, w, None, [ctx.stride] * 2, [ctx.pad] * 2, [1, 1], False, [0, 0], 1,
                                                         [True, False, False])[0]
        if ctx.needs_input_grad[1]:
            g = getattr(ctx.w_ref, "grad", None)
            gv = g.permute(0, 2, 3, 1) if (g is not None and g.dtype == torch.bfloat16 and g.dim() == 4) else None
            if gv is not None and gv.is_contiguous():
                conv_wgrad_nhwc(x, dy, w.shape, ctx.stride, ctx.pad, out=gv, accumulate=True)   # straight into the flat gradient buffer
            else:
                dw = conv_wgrad_nhwc(x, dy, w.shape, ctx.stride, ctx.pad)
        return dx, dw, None, None, None


def conv_nhwc(x: torch.Tensor, w: torch.Tensor, stride: int = 1, pad: int = 1, want_stats: bool = False):
    return _ConvNHWC.apply(x, w, stride, pad, want_stats)


# ---- ResNet stem: dense 4x4 convolution over the 16-channel space-to-depth input (native/gemm/stem_s2d.inc) --------------------------
def stem_s2d_ok(x: torch.Tensor, w2: torch.Tensor) -> bool:
    """x: [N,16,Hp,Wp] channels_last bf16 (the s2d input of ops.fused.u8_to_s2d_norm), w2: [64,16,4,4]."""
    return (x.is_cuda and x.dtype == torch.bfloat16 and x.dim() == 4 and x.shape[1] == 16 and tuple(w2.shape) == (64, 16, 4, 4)
            and 4 <= x.shape[3] <= 128 and x.shape[2] >= 4)


def stem_s2d_fprop(x: torch.Tensor, w2: torch.Tensor, stats: Optional[torch.Tensor] = None, max_ctas: int = 0) -> torch.Tensor:
    """y[N,64,Hp-3,Wp-3] (channels_last) = conv2d(x, w2) on the tcgen05 stem kernel: one output row per tile, the 16 filter taps as
    row-shifted 32-byte-swizzle descriptors over four TMA-loaded input rows, weights stationary in shared memory.
    stats: zero-initialised float32[128] receiving the per-channel sum / sum of squares of y (train-mode BatchNorm statistics)."""
    n, _, hp, wp = x.shape
    xs, ws_ = _nhwc_storage(x), _nhwc_storage(w2)
    y = torch.empty((n, hp - 3, wp - 3, 64), dtype=torch.bfloat16, device=x.device)
    lib = load()
    rc = lib.sy_stem_s2d_fprop(C.c_void_p(xs.data_ptr()), C.c_void_p(ws_.data_ptr()), C.c_void_p(y.data_ptr()), n, hp, wp,
                               C.c_void_p(stats.data_ptr() if stats is not None else 0), max_ctas,
                               C.c_void_p(torch.cuda.current_stream(x.device).cuda_stream))
    if rc != 0:
        raise RuntimeError(f"sy_stem_s2d_fprop failed ({rc}): {lib.sy_gemm_last_error().decode()}")
    return y.permute(0, 3, 1, 2)


def stem_s2d_wgrad(x: torch.Tensor, dy: torch.Tensor, out: Optional[torch.Tensor] = None, accumulate: bool = False,
                   max_ctas: int = 0) -> torch.Tensor:
    """dW2[64,16,4,4] (stored [64][4][4][16]) of the stem convolution: X rows as MN-major operands whose slabs are one pixel apart (the
    four horizontal taps of a filter row come out of ONE buffer), dY rows as the B operand, accumulators resident in TMEM for all
    tiles of a CTA, cross-CTA reduction through the fp32 workspace (last CTA converts to bf16)."""
    n, _, hp, wp = x.shape
    xs, dys = _nhwc_storage(x), _nhwc_storage(dy)
    assert tuple(dys.shape) == (n, hp - 3, wp - 3, 64), dys.shape
    if out is None:
        out = torch.empty((64, 4, 4, 16), dtype=torch.bfloat16, device=x.device)
        accumulate = False
    assert out.is_contiguous() and tuple(out.shape) == (64, 4, 4, 16) and out.dtype == torch.bfloat16
    ws, tickets = _workspace(x.device)
    lib = load()
    rc = lib.sy_stem_s2d_wgrad(C.c_void_p(xs.data_ptr()), C.c_void_p(dys.data_ptr()), C.c_void_p(out.data_ptr()), n, hp, wp,
                               C.c_void_p(ws.data_ptr()), C.c_void_p(tickets.data_ptr()), 1 if accumulate else 0, max_ctas,
                               C.c_void_p(torch.cuda.current_stream(x.device).cuda_stream))
    if rc != 0:
        raise RuntimeError(f"sy_stem_s2d_wgrad failed ({rc}): {lib.sy_gemm_last_error().decode()}")
    return out.permute(0, 3, 1, 2)


class _StemS2D(torch.autograd.Function):
    """Stem convolution on the s2d input: fprop (+ BatchNorm statistics) and wgrad on tcgen05; the input needs no gradient."""

    @staticmethod
    def forward(ctx, x, w2, want_stats):
        ctx.set_materialize_grads(False)          # the statistics output has no gradient: do not let autograd build a zeros tensor for it
        stats = _pool_zeros(128, x.device) if want_stats else None
        y = stem_s2d_fprop(x, w2, stats=stats)
        ctx.save_for_backward(x)
        if stats is not None:
            ctx.mark_non_differentiable(stats)
        return y, stats

    @staticmethod
    def backward(ctx, dy, _ds):
        (x,) = ctx.saved_tensors
        if not dy.is_contiguous(memory_format=torch.channels_last):
            dy = dy.contiguous(memory_format=torch.channels_last)
        return None, stem_s2d_wgrad(x, dy), None


def stem_conv_s2d(x: torch.Tensor, w2: torch.Tensor, want_stats: bool = True):
    """(y, stats) of the s2d stem convolution; stats is None when not requested."""
    return _StemS2D.apply(x, w2, want_stats)


# ---- inference: BatchNorm folded into the GEMM / convolution epilogue ------------------------------------------------------------
def conv_affine_ok(x: torch.Tensor, w: torch.Tensor, stride: int) -> bool:
    """Shapes ``conv_affine_nhwc`` accepts: 1x1 / stride 1 as a GEMM (channels % 8), anything else through the im2col kernel
    (input channels % 64, output channels % 8, N*P*Q % 128)."""
    if not (x.is_cuda and x.dtype == torch.bfloat16 and w.dtype == torch.bfloat16):
        return False
    cin, cout, k = x.shape[1], w.shape[0], w.shape[2]
    if k == 1 and stride == 1:
        return cin % 8 == 0 and cout % 8 == 0
    return conv_supported(x, w, stride, k // 2)


def conv_affine_nhwc(x: torch.Tensor, w: torch.Tensor, scale: torch.Tensor, shift: torch.Tensor, stride: int = 1,
                     residual: Optional[torch.Tensor] = None, relu: bool = True, block_n: int = 0, max_ctas: int = 0) -> torch.Tensor:
    """y = act(conv2d(x, w, stride, 'same') * scale + shift (+ residual)) for channels_last bf16 x[N,Cin,H,W], w[Cout,Cin,K,K] (stored
    KRSC), fp32 scale / shift [Cout], optional channels_last bf16 residual shaped like y: the inference form of conv + BatchNorm
    (+ residual add) (+ ReLU) in ONE tcgen05 kernel, accumulator scaled in fp32 and rounded to bf16 once.  1x1 / stride 1 runs as the
    GEMM, everything else as the TMA-im2col convolution.  Returns channels_last y."""
    n, cin, h, wd = x.shape
    cout, _, r, s = w.shape
    pad = r // 2
    p, q = (h + 2 * pad - r) // stride + 1, (wd + 2 * pad - s) // stride + 1
    assert x.is_cuda and x.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and w.shape[1] == cin and r == s
    assert scale.dtype == torch.float32 and shift.dtype == torch.float32 and scale.numel() == cout and shift.numel() == cout
    assert scale.is_contiguous() and shift.is_contiguous()
    assert cout % 8 == 0, "conv_affine_nhwc: output channels % 8"
    xs, ws = _nhwc_storage(x), _nhwc_storage(w)
    rs = None
    if residual is not None:
        assert tuple(residual.shape) == (n, cout, p, q) and residual.dtype == torch.bfloat16
        rs = _nhwc_storage(residual)
    y = torch.empty((n, p, q, cout), dtype=torch.bfloat16, device=x.device)
    lib = load()
    stream = C.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)
    rptr = C.c_void_p(rs.data_ptr() if rs is not None else 0)
    if r == 1 and stride == 1:
        assert cin % 8 == 0, "1x1 GEMM: input channels % 8"
        rc = lib.sy_gemm_bf16_tn_affine(C.c_void_p(xs.data_ptr()), C.c_void_p(ws.data_ptr()), C.c_void_p(y.data_ptr()), n * h * wd, cout, cin,
                                        cin, cin, cout, C.c_void_p(scale.data_ptr()), C.c_void_p(shift.data_ptr()), rptr, cout,
                                        1 if relu else 0, block_n, max_ctas, stream)
        if rc != 0:
            raise RuntimeError(f"sy_gemm_bf16_tn_affine failed ({rc}): {lib.sy_gemm_last_error().decode()}")
    else:
        assert conv_supported(x, w, stride, pad), "conv_affine_nhwc: input channels % 64 and N*P*Q % 128 for the im2col kernel"
        rc = lib.sy_conv_bf16_nhwc_affine(C.c_void_p(xs.data_ptr()), C.c_void_p(ws.data_ptr()), C.c_void_p(y.data_ptr()), n, h, wd, cin, cout,
                                          r, s, pad, stride, C.c_void_p(scale.data_ptr()), C.c_void_p(shift.data_ptr()), rptr,
                                          1 if relu else 0, block_n, max_ctas, stream)
        if rc != 0:
            raise RuntimeError(f"sy_conv_bf16_nhwc_affine failed ({rc}): {lib.sy_gemm_last_error().decode()}")
    return y.permute(0, 3, 1, 2)
