"""ctypes binding for ``libshipyard_ops`` (fused elementwise / normalisation kernels).

No counterpart in the reference: its recipes run framework containers (e.g. MNIST on PyTorch,
/root/reference/recipes/PyTorch-GPU/config/jobs.yaml:1-8); these kernels are the memory-bound half of the
retargeted ResNet-50 recipe (BN(+residual)(+ReLU) forward / backward, max-pool, uint8 -> bf16 input conversion)
and of the HPCG retarget (``sy_hpcg_*``, /root/reference/recipes/HPCG-Infiniband-IntelMPI/config/docker/jobs.yaml:5-20).
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_LIB = None
IMAGENET_MEAN = (0.485, 0.456, 0.406)
IMAGENET_STD = (0.229, 0.224, 0.225)


def lib_path() -> str:
    return os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "_native", "libshipyard_ops.so")


def load() -> C.CDLL:
    global _LIB
    if _LIB is None:
        p = lib_path()
        if not os.path.exists(p):
            from .._build import ensure_built
            ensure_built(["ops"])
        if not os.path.exists(p):
            raise RuntimeError(f"{p} missing: run `python native/build.py ops` (no Python fallback on GPU)")
        lib = C.CDLL(p)
        lib.sy_ops_launch_count.restype = C.c_ulonglong
        lib.sy_ops_u8_to_bf16_norm.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_float),
                                               C.POINTER(C.c_float), C.c_void_p]
        _LIB = lib
    return _LIB


def launch_count() -> int:
    return int(load().sy_ops_launch_count())


def _stream(t: torch.Tensor) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def u8_to_bf16_norm(src_u8: torch.Tensor, dst_bf16: torch.Tensor, mean=IMAGENET_MEAN, std=IMAGENET_STD) -> torch.Tensor:
    """uint8 NHWC (C=3) -> normalised bf16 NHWC, one pass, on ``dst``'s current stream."""
    assert src_u8.dtype == torch.uint8 and dst_bf16.dtype == torch.bfloat16
    assert src_u8.numel() == dst_bf16.numel() and src_u8.is_cuda and dst_bf16.is_cuda
    m = (C.c_float * 3)(*mean)
    s = (C.c_float * 3)(*std)
    rc = load().sy_ops_u8_to_bf16_norm(C.c_void_p(src_u8.data_ptr()), C.c_void_p(dst_bf16.data_ptr()),
                                       src_u8.numel(), m, s, _stream(dst_bf16))
    if rc != 0:
        raise RuntimeError(f"u8_to_bf16_norm launch failed: cuda error {rc}")
    return dst_bf16


# ---------------------------------------------------------------------------
# fused train-mode BatchNorm (+ residual) (+ ReLU), NHWC bf16
# ---------------------------------------------------------------------------
def _bind_bn(lib):
    if getattr(lib, "_bn_bound", False):
        return
    vp, fp = C.c_void_p, C.c_void_p
    lib.sy_ops_bn_fwd.argtypes = [vp, vp, vp, vp, vp, fp, fp, fp, fp, fp, C.c_long, C.c_int, C.c_float, C.c_float,
                                  C.c_int, vp, vp]
    lib.sy_ops_bn_apply_only.argtypes = [vp, vp, vp, vp, vp, fp, fp, fp, fp, fp, C.c_long, C.c_int, C.c_float,
                                         C.c_float, C.c_int, vp, vp]
    lib.sy_ops_bn_bwd.argtypes = [vp, vp, vp, fp, fp, vp, vp, vp, vp, vp, fp, C.c_long, C.c_int, C.c_int, C.c_int, vp, vp]
    lib.sy_ops_set_ws_prezeroed.argtypes = [C.c_int]
    lib.sy_ops_bn_bwd_dual.argtypes = [vp, vp, vp, fp, fp, vp, vp, vp, vp, vp, fp, C.c_long, C.c_int, C.c_int, C.c_int, vp, vp]
    lib.sy_ops_maxpool3x3s2_fwd.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp]
    lib.sy_ops_maxpool3x3s2_bwd.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp]
    lib.sy_ops_u8_to_s2d_norm.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float), vp]
    lib.sy_ops_bn_fold.argtypes = [vp, C.c_int, vp]
    lib.sy_ops_bn_infer_apply.argtypes = [vp, vp, vp, fp, fp, C.c_long, C.c_int, C.c_int, vp]
    lib._bn_bound = True


def _ptr(t):
    return C.c_void_p(0 if t is None else t.data_ptr())


def _is_nhwc(t: torch.Tensor) -> bool:
    return t.dim() == 4 and t.permute(0, 2, 3, 1).is_contiguous()


def bn_shape_supported(c: int) -> bool:
    g = c // 8
    return c % 8 == 0 and 1 <= g <= 256 and (g & (g - 1)) == 0


# ---- zero pool: ONE memset per training step instead of one per layer -------------------------------------------------------------
# Every fused BN layer needs a zeroed float[2C] scratch in forward (statistics) and in backward (reductions), and every GEMM with fused
# statistics a zeroed float[2C] output: ~100 torch.zeros / cudaMemsetAsync nodes of a few hundred bytes each per ResNet-50 step
# (0.24 ms of launch-bound work in the captured graph, gpurun_out/c6_kernel_census.txt).  The trainer opens a pool at the start of the
# step (one memset of the whole arena); zeros(n) then hands out consecutive slices.  Outside a pool everything behaves as before.
_ZPOOL: dict = {"buf": None, "off": 0, "active": False}


def zero_pool_begin(device, nfloats: int = 1 << 18) -> None:
    if not (isinstance(device, torch.device) and device.type == "cuda"):
        return
    buf = _ZPOOL["buf"]
    if buf is None or buf.device != device or buf.numel() < nfloats:
        buf = _ZPOOL["buf"] = torch.empty(nfloats, dtype=torch.float32, device=device)
    buf.zero_()
    _ZPOOL.update(off=0, active=True)
    lib = load(); _bind_bn(lib)
    lib.sy_ops_set_ws_prezeroed(1)


def zero_pool_end() -> None:
    _ZPOOL["active"] = False
    if _LIB is not None:
        _LIB.sy_ops_set_ws_prezeroed(0)


def zeros(n: int, device) -> torch.Tensor:
    """float32 zeros: a slice of the step's zero pool when one is open (and has room), else a fresh torch.zeros."""
    buf = _ZPOOL["buf"]
    n_al = (n + 31) // 32 * 32                            # 128-byte aligned slices
    if _ZPOOL["active"] and buf is not None and buf.device == device and _ZPOOL["off"] + n_al <= buf.numel():
        o = _ZPOOL["off"]
        _ZPOOL["off"] = o + n_al
        return buf[o:o + n]
    if _ZPOOL["active"]:
        z = torch.zeros(n, dtype=torch.float32, device=device)      # pool exhausted: correct, just not free
        return z
    return torch.zeros(n, dtype=torch.float32, device=device)


def _scratch(n: int, device) -> torch.Tensor:
    """float[n] scratch the BN kernels expect zeroed: pool slice inside a step (kernels skip their memset), plain empty otherwise."""
    if _ZPOOL["active"]:
        return zeros(n, device)
    return torch.empty(n, dtype=torch.float32, device=device)


class _FusedBNAct(torch.autograd.Function):
    """y = act(BN_train(x) [+ residual]) with saved (x, y, mean, invstd) for the fused backward."""

    @staticmethod
    def forward(ctx, x, gamma, beta, residual, running_mean, running_var, relu, eps, momentum, stats, dual=False):
        lib = load(); _bind_bn(lib)
        ctx.set_materialize_grads(False)                # an unused second output must arrive as None, not as a zeros tensor
        assert x.is_cuda and x.dtype == torch.bfloat16 and _is_nhwc(x), "fused BN wants NHWC bf16"
        n, c, h, w = x.shape
        m = n * h * w
        out = torch.empty_like(x)                       # preserves channels_last strides
        save_mean = torch.empty(c, dtype=torch.float32, device=x.device)
        save_invstd = torch.empty(c, dtype=torch.float32, device=x.device)
        if residual is not None:
            assert residual.shape == x.shape and _is_nhwc(residual) and residual.dtype == x.dtype
        # ReLU sign bits (1 bit / element) saved for backward instead of re-reading the activation
        mask = torch.empty(m * (c // 8), dtype=torch.uint8, device=x.device) if relu else None
        if stats is None:
            ws = _scratch(2 * c, x.device)
            rc = lib.sy_ops_bn_fwd(_ptr(x), _ptr(residual), _ptr(out), _ptr(gamma), _ptr(beta), _ptr(running_mean),
                                   _ptr(running_var), _ptr(save_mean), _ptr(save_invstd), _ptr(ws), m, c, eps,
                                   momentum, 1 if relu else 0, _ptr(mask), _stream(x))
        else:
            rc = lib.sy_ops_bn_apply_only(_ptr(x), _ptr(residual), _ptr(out), _ptr(gamma), _ptr(beta),
                                          _ptr(running_mean), _ptr(running_var), _ptr(save_mean), _ptr(save_invstd),
                                          _ptr(stats), m, c, eps, momentum, 1 if relu else 0, _ptr(mask), _stream(x))
        if rc != 0:
            raise RuntimeError(f"fused BN forward failed (rc={rc}, C={c})")
        ctx.save_for_backward(x, mask if mask is not None else save_mean, save_mean, save_invstd, gamma)
        ctx.has_mask = mask is not None
        ctx.relu, ctx.has_res = bool(relu), residual is not None
        ctx.beta_ref = beta if isinstance(beta, torch.nn.Parameter) else None
        ctx.dual = bool(dual)
        if dual:
            # the same activation twice: consumers that use the two handles (next block's first conv / its residual input)
            # send their gradients back separately, and the backward kernels add them in registers (no add kernel)
            return out, out.view_as(out)
        return out

    @staticmethod
    def backward(ctx, dout, dout2=None):
        lib = load(); _bind_bn(lib)
        x, mask, mean, invstd, gamma = ctx.saved_tensors
        mask = mask if ctx.has_mask else None
        n, c, h, w = x.shape
        m = n * h * w
        nres = 11
        if dout is None:
            dout, dout2 = dout2, None
        if dout is None:
            return (None,) * nres
        if not _is_nhwc(dout):
            dout = dout.contiguous(memory_format=torch.channels_last)
        if dout2 is not None and not _is_nhwc(dout2):
            dout2 = dout2.contiguous(memory_format=torch.channels_last)
        if dout2 is not None and ctx.relu and mask is None:
            dout, dout2 = dout + dout2, None            # the two-gradient kernels gate with the bit mask only
        dx = torch.empty_like(x)
        dres = torch.empty_like(x) if ctx.has_res else None
        # write dgamma/dbeta straight into the parameters' .grad views when they exist (flat gradient buffer):
        # saves two AccumulateGrad add-kernels per layer
        beta = ctx.beta_ref
        direct = (isinstance(gamma, torch.nn.Parameter) and gamma.grad is not None and beta is not None and beta.grad is not None
                  and gamma.grad.is_contiguous() and beta.grad.is_contiguous())
        if direct:
            dgamma, dbeta = gamma.grad, beta.grad
        else:
            dgamma = torch.empty(c, dtype=torch.bfloat16, device=x.device)
            dbeta = torch.empty(c, dtype=torch.bfloat16, device=x.device)
        ws = _scratch(2 * c, x.device)
        if dout2 is not None:
            rc = lib.sy_ops_bn_bwd_dual(_ptr(dout), _ptr(dout2), _ptr(x), _ptr(mean), _ptr(invstd), _ptr(gamma), _ptr(dx),
                                        _ptr(dres), _ptr(dgamma), _ptr(dbeta), _ptr(ws), m, c, 1 if ctx.relu else 0,
                                        1 if direct else 0, _ptr(mask), _stream(x))
        else:
            rc = lib.sy_ops_bn_bwd(_ptr(dout), None, _ptr(x), _ptr(mean), _ptr(invstd), _ptr(gamma), _ptr(dx),
                                   _ptr(dres), _ptr(dgamma), _ptr(dbeta), _ptr(ws), m, c, 1 if ctx.relu else 0,
                                   1 if direct else 0, _ptr(mask), _stream(x))
        if rc != 0:
            raise RuntimeError(f"fused BN backward failed (rc={rc})")
        if direct:
            return (dx, None, None, dres) + (None,) * (nres - 4)
        return (dx, dgamma, dbeta, dres) + (None,) * (nres - 4)


def fused_bn_act(x, gamma, beta, residual=None, running_mean=None, running_var=None, relu=True, eps=1e-5,
                 momentum=0.1, stats=None, dual=False):
    """Train-mode BN + optional residual + optional ReLU in two passes (NHWC bf16, CUDA only).

    ``dual=True`` returns the output twice ``(y, y_alias)`` (same storage): give one handle to each of two consumers and
    their gradients are summed inside the backward kernels instead of by a separate autograd add kernel."""
    return _FusedBNAct.apply(x, gamma, beta, residual, running_mean, running_var, relu, eps, momentum, stats, dual)


def bn_act_reference(x, gamma, beta, residual=None, relu=True, eps=1e-5):
    """Plain PyTorch fp32 reference of the same op (used by the numerics tests and the CPU path)."""
    xf = x.float()
    mean = xf.mean(dim=(0, 2, 3), keepdim=True)
    var = xf.var(dim=(0, 2, 3), unbiased=False, keepdim=True)
    y = (xf - mean) * torch.rsqrt(var + eps) * gamma.float().view(1, -1, 1, 1) + beta.float().view(1, -1, 1, 1)
    if residual is not None:
        y = y + residual.float()
    return torch.relu(y) if relu else y


# ---------------------------------------------------------------------------
# max-pool 3x3/s2/p1 (NHWC bf16) with saved arg-max codes
# ---------------------------------------------------------------------------
class _MaxPool3x3s2(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        lib = load(); _bind_bn(lib)
        assert x.is_cuda and x.dtype == torch.bfloat16 and _is_nhwc(x) and x.shape[1] % 8 == 0
        n, c, h, w = x.shape
        oh, ow = (h + 2 - 3) // 2 + 1, (w + 2 - 3) // 2 + 1
        y = torch.empty((n, oh, ow, c), dtype=x.dtype, device=x.device).permute(0, 3, 1, 2)
        idx = torch.empty((n, oh, ow, c), dtype=torch.uint8, device=x.device)
        rc = lib.sy_ops_maxpool3x3s2_fwd(_ptr(x), _ptr(y), _ptr(idx), n, h, w, c, _stream(x))
        if rc != 0:
            raise RuntimeError(f"maxpool forward failed ({rc})")
        ctx.save_for_backward(idx)
        ctx.shape = (n, c, h, w)
        return y

    @staticmethod
    def backward(ctx, dy):
        lib = load()
        (idx,) = ctx.saved_tensors
        n, c, h, w = ctx.shape
        if not _is_nhwc(dy):
            dy = dy.contiguous(memory_format=torch.channels_last)
        dx = torch.empty((n, h, w, c), dtype=dy.dtype, device=dy.device).permute(0, 3, 1, 2)
        rc = lib.sy_ops_maxpool3x3s2_bwd(_ptr(dy), _ptr(idx), _ptr(dx), n, h, w, c, _stream(dy))
        if rc != 0:
            raise RuntimeError(f"maxpool backward failed ({rc})")
        return dx


def maxpool3x3s2(x: torch.Tensor) -> torch.Tensor:
    return _MaxPool3x3s2.apply(x)


def maxpool3x3s2_infer(x: torch.Tensor) -> torch.Tensor:
    """Inference max-pool 3x3/s2/p1 on channels_last bf16 (no arg-max codes: nothing is kept for a backward pass)."""
    lib = load(); _bind_bn(lib)
    assert x.is_cuda and x.dtype == torch.bfloat16 and _is_nhwc(x) and x.shape[1] % 8 == 0
    n, c, h, w = x.shape
    oh, ow = (h + 2 - 3) // 2 + 1, (w + 2 - 3) // 2 + 1
    y = torch.empty((n, oh, ow, c), dtype=x.dtype, device=x.device).permute(0, 3, 1, 2)
    rc = lib.sy_ops_maxpool3x3s2_fwd(_ptr(x), _ptr(y), None, n, h, w, c, _stream(x))
    if rc != 0:
        raise RuntimeError(f"maxpool (inference) failed ({rc})")
    return y


# ---------------------------------------------------------------------------
# inference BatchNorm: folded per-channel affine maps
# ---------------------------------------------------------------------------
def bn_fold_reference(gamma, beta, running_mean, running_var, eps=1e-5):
    """(scale, shift) in fp32 with BN_eval(x) = x * scale + shift: the formula the fold kernel computes."""
    scale = gamma.float() * torch.rsqrt(running_var.float() + eps)
    return scale, beta.float() - running_mean.float() * scale


class BnFoldTable:
    """Device table for ``bn_fold``: one 64-byte entry {gamma, beta, running_mean, running_var, scale_out, shift_out, C, eps} per BN
    layer, and the fp32 scale / shift outputs (every layer's slice 32-byte aligned for the 16-byte vector loads of the consumers).

    The entries hold raw pointers to the parameters and statistics: the table stays valid while those tensors keep their storage."""

    def __init__(self, layers, device):
        """layers: list of (gamma bf16[C], beta bf16[C], running_mean fp32[C], running_var fp32[C], eps)."""
        import struct
        offs, total = [], 0
        for g, b, m, v, _ in layers:
            c = g.numel()
            assert g.dtype == torch.bfloat16 and b.dtype == torch.bfloat16, "bn_fold: gamma / beta must be bf16"
            assert m.dtype == torch.float32 and v.dtype == torch.float32, "bn_fold: running statistics must be fp32"
            assert all(t.is_cuda and t.is_contiguous() and t.numel() == c for t in (g, b, m, v))
            offs.append(total)
            total += (c + 7) // 8 * 8
        self.buf = torch.zeros(2, max(total, 8), dtype=torch.float32, device=device)
        self.scale = [self.buf[0, o:o + g.numel()] for o, (g, *_r) in zip(offs, layers)]
        self.shift = [self.buf[1, o:o + g.numel()] for o, (g, *_r) in zip(offs, layers)]
        words = []
        for (g, b, m, v, eps), sc, sh in zip(layers, self.scale, self.shift):
            eps_bits = struct.unpack("<I", struct.pack("<f", float(eps)))[0]
            words += [g.data_ptr(), b.data_ptr(), m.data_ptr(), v.data_ptr(), sc.data_ptr(), sh.data_ptr(), g.numel(), eps_bits]
        self.table = torch.tensor(words, dtype=torch.int64).to(device)
        self.n_layers = len(layers)
        self._keep = layers                       # the pointed-to tensors must outlive the table


def bn_fold(table: BnFoldTable) -> None:
    """scale = gamma * rsqrt(running_var + eps), shift = beta - running_mean * scale for every layer of ``table``: ONE launch."""
    lib = load(); _bind_bn(lib)
    rc = lib.sy_ops_bn_fold(_ptr(table.table), table.n_layers, _stream(table.table))
    if rc != 0:
        raise RuntimeError(f"bn_fold failed ({rc})")


def bn_infer_apply(x: torch.Tensor, scale: torch.Tensor, shift: torch.Tensor, residual=None, relu: bool = True,
                   out=None) -> torch.Tensor:
    """out = act(x * scale + shift (+ residual)) on channels_last bf16 (inference BatchNorm of a layer whose convolution has no
    fused epilogue).  ``out`` may be ``x`` (in place)."""
    lib = load(); _bind_bn(lib)
    assert x.is_cuda and x.dtype == torch.bfloat16 and _is_nhwc(x), "bn_infer_apply wants channels_last bf16"
    n, c, h, w = x.shape
    assert c % 8 == 0, "bn_infer_apply: channels % 8"
    assert scale.dtype == torch.float32 and shift.dtype == torch.float32 and scale.numel() == c and shift.numel() == c
    if residual is not None:
        assert residual.shape == x.shape and residual.dtype == x.dtype and _is_nhwc(residual)
    out = torch.empty_like(x) if out is None else out
    assert out.shape == x.shape and _is_nhwc(out)
    rc = lib.sy_ops_bn_infer_apply(_ptr(x), _ptr(residual), _ptr(out), _ptr(scale), _ptr(shift), n * h * w, c, 1 if relu else 0,
                                   _stream(x))
    if rc != 0:
        raise RuntimeError(f"bn_infer_apply failed ({rc})")
    return out


def u8_to_s2d_norm(src_u8: torch.Tensor, dst: torch.Tensor, mean=IMAGENET_MEAN, std=IMAGENET_STD) -> torch.Tensor:
    """uint8 NHWC [N,H,W,3] -> normalised, zero-bordered space-to-depth bf16 [N,H/2+3,W/2+3,16] (stem input)."""
    lib = load(); _bind_bn(lib)
    n, h, w, c = src_u8.shape
    assert c == 3 and src_u8.dtype == torch.uint8 and dst.dtype == torch.bfloat16 and dst.is_contiguous()
    assert tuple(dst.shape) == (n, h // 2 + 3, w // 2 + 3, 16), dst.shape
    m = (C.c_float * 3)(*mean); s = (C.c_float * 3)(*std)
    rc = lib.sy_ops_u8_to_s2d_norm(_ptr(src_u8), _ptr(dst), n, h, w, m, s, _stream(dst))
    if rc != 0:
        raise RuntimeError(f"u8_to_s2d_norm failed ({rc})")
    return dst


def s2d_reference(x_nchw: torch.Tensor) -> torch.Tensor:
    """PyTorch reference of the stem input transform: [N,3,H,W] float -> [N,16,H/2+3,W/2+3] (zero border/channels)."""
    n, c, h, w = x_nchw.shape
    t = x_nchw.view(n, c, h // 2, 2, w // 2, 2).permute(0, 3, 5, 1, 2, 4).reshape(n, 12, h // 2, w // 2)   # (p,q,c)
    out = x_nchw.new_zeros((n, 16, h // 2 + 3, w // 2 + 3))
    out[:, :12, 2:2 + h // 2, 2:2 + w // 2] = t
    return out


def stem_weight_s2d(w: torch.Tensor) -> torch.Tensor:
    """[Cout,3,7,7] stride-2 pad-3 kernel -> equivalent [Cout,16,4,4] stride-1 kernel over the s2d input."""
    co = w.shape[0]
    w8 = torch.nn.functional.pad(w, (1, 0, 1, 0))                       # ky' = ky + 1 (zero row/col first)
    w2 = w8.reshape(co, 3, 4, 2, 4, 2).permute(0, 3, 5, 1, 2, 4).reshape(co, 12, 4, 4)   # channel = (p*2+q)*3 + c
    return torch.nn.functional.pad(w2, (0, 0, 0, 0, 0, 4))
