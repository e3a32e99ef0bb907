"""Convolution dispatcher: per layer shape and per pass (fprop / dgrad / wgrad) pick the faster of the tcgen05
implicit-GEMM kernels (``ops.gemm``) and cuDNN, from timings taken on the device the first time a shape is seen.

The reference has no compute path at all (its recipes run third-party framework containers,
/root/reference/recipes/PyTorch-GPU/config/jobs.yaml:1-8); this is part of the retargeted ResNet-50 recipe.

``SHIPYARD_CONV_IMPL`` = ``auto`` (default: measure, keep the faster), ``tc`` (always our kernels where the shape is
supported) or ``cudnn`` (library only).  The chosen table is available from ``plan_table()`` and is printed by bench.py.

``SHIPYARD_CONV_HALO`` (default on; ``0`` removes them) adds the halo-load 3x3 kernels (``th`` / ``th2``, native/gemm/conv_halo.inc: one TMA box per tile and
channel block instead of nine im2col boxes) to the candidates.  Every halo candidate is first compared against the cuDNN
result of the same call; a mismatch disables the halo kernels for the process (``halo_state()``) instead of training on them.
"""
from __future__ import annotations

import os
from dataclasses import dataclass, asdict
from typing import Optional

import torch
import torch.nn.functional as F

from . import gemm as _gemm
from .fused import zeros as _fused_zeros

_MODE = os.environ.get("SHIPYARD_CONV_IMPL", "auto").lower()
_PLANS: dict = {}
_HALO = os.environ.get("SHIPYARD_CONV_HALO", "1") not in ("0", "", "off", "false")
# The additional halo variants (alternate-tile epilogue, 64-column CTA pairs, weights-stationary pair kernel, halo-load wgrad) passed
# their numerics tests on hardware in round 2 (tests/test_gpu_conv_halo.py) and take part in the race by default; every one of them
# must still reproduce the cuDNN result of the same call first (_halo_check).  SHIPYARD_CONV_EXPERIMENTAL=0 removes them, a comma
# list restricts them, e.g. SHIPYARD_CONV_EXPERIMENTAL=tha,wgrad_th (names: tha th264 th264a th2w wgrad_th).
_EXP_RAW = os.environ.get("SHIPYARD_CONV_EXPERIMENTAL", "1")
_EXP = _EXP_RAW not in ("0", "", "off", "false")
_EXP_ALLOW = None if _EXP_RAW in ("0", "", "off", "false", "1", "on", "true", "all") else {v.strip() for v in _EXP_RAW.split(",") if v.strip()}
# impl name -> keyword arguments of ops.gemm.conv3x3_halo
_HALO_KW = {"th": {}, "th2": {"pair": True}, "tha": {"epi_alt": True}, "th264": {"pair": True, "block_n": 64},
            "th264a": {"pair": True, "block_n": 64, "epi_alt": True}, "th2w": {"pair": True, "weights_stationary": True}}
_HALO_STATE = {"enabled": _HALO, "checked": 0, "failed": []}
_HBM_BPS = 5.4e12          # measured bandwidth of the stand-alone BN statistics pass (profiles/ncu_bn_kernels.md)


@dataclass
class ConvPlan:
    fprop: str = "cudnn"      # "tc" (1-CTA tcgen05 im2col) | "tc2" (CTA pair) | "th" (halo load) | "th2" (halo, CTA pair) | "cudnn"
    #                           experimental (SHIPYARD_CONV_EXPERIMENTAL): "tha" | "th264" | "th264a" | "th2w" (see _HALO_KW); wgrad "th"
    dgrad: str = "cudnn"
    wgrad: str = "cudnn"
    stats: bool = False       # fprop produces the BatchNorm statistics in its epilogue
    timings_us: Optional[dict] = None


# Tie-break of the race: an own kernel within this fraction of the library's time wins.  The race's own repeatability was measured by
# running it twice in one process (gpurun_out/c6_bench.err, "rerace"): the SAME cuDNN kernel on the same shape differs by up to 3.6 %
# between the two runs (158.7 vs 164.5 us), ours by up to 1.2 %.  Inside a 5 % band "faster" is therefore noise and the native kernel is
# preferred; SHIPYARD_CONV_TIE=0 gives the strict race.
_TIE = float(os.environ.get("SHIPYARD_CONV_TIE", "0.05"))


def _pick(t: dict, prefix: str) -> str:
    """Winner among the timings whose key starts with `prefix` ('fprop_' / 'dgrad_' / 'wgrad_'), native-preferring inside the tie band."""
    keys = [k for k in t if k.startswith(prefix)]
    own = [k for k in keys if not k.startswith(prefix + "cudnn")]
    lib = [k for k in keys if k.startswith(prefix + "cudnn")]
    best_own = min(own, key=lambda k: t[k]) if own else None
    best_lib = min(lib, key=lambda k: t[k]) if lib else None
    if best_own is None:
        return best_lib
    if best_lib is None or t[best_own] <= t[best_lib] * (1.0 + _TIE):
        return best_own
    return best_lib


_STEM = os.environ.get("SHIPYARD_STEM_IMPL", "tc").lower()          # "tc": native/gemm/stem_s2d.inc; "cudnn": F.conv2d on the s2d input


def stem_native() -> bool:
    """The s2d stem runs on the repo's tcgen05 kernels unless SHIPYARD_STEM_IMPL=cudnn or the dispatcher is forced to cuDNN."""
    return _STEM != "cudnn" and _MODE != "cudnn"


def set_stem(impl: str) -> None:
    global _STEM
    assert impl in ("tc", "cudnn")
    _STEM = impl


def set_mode(mode: str) -> None:
    global _MODE
    assert mode in ("auto", "tc", "cudnn")
    _MODE = mode
    _PLANS.clear()
    _INFER_PLANS.clear()


def set_halo(on: bool) -> None:
    """Enable / disable the halo-load 3x3 candidates (clears the plan table)."""
    _HALO_STATE.update(enabled=bool(on), checked=0, failed=[])
    _PLANS.clear()


def halo_state() -> dict:
    return dict(_HALO_STATE)


def plan_table() -> dict:
    return {"x".join(map(str, k)): {kk: vv for kk, vv in asdict(v).items()} for k, v in _PLANS.items()}


def _key(x: torch.Tensor, w: torch.Tensor, stride: int):
    n, cin, h, wd = x.shape
    return (n, cin, h, wd, w.shape[0], w.shape[2], stride)


def _tc_caps(x: torch.Tensor, w: torch.Tensor, stride: int) -> dict:
    """Which passes the tcgen05 kernels support for this shape."""
    n, cin, h, wd = x.shape
    cout, _, k, _ = w.shape
    pad = k // 2
    ok = x.is_cuda and x.dtype == torch.bfloat16
    if k == 1 and stride == 1:
        g = ok and cin % 8 == 0 and cout % 8 == 0
        return {"fprop": g, "dgrad": g, "wgrad": g}
    sup = ok and _gemm.conv_supported(x, w, stride, pad)
    # 1x1 / stride-2 (downsample branches): the data gradient is a GEMM with a scattering epilogue (ops.gemm.conv1x1_s2_dgrad)
    s2_1x1 = ok and k == 1 and stride == 2 and h % 2 == 0 and wd % 2 == 0 and cin % 8 == 0 and cout % 8 == 0
    return {"fprop": sup, "wgrad": sup, "dgrad": (sup and stride == 1 and cout % 64 == 0) or s2_1x1}


def _time(fn, iters: int = 5, reps: int = 4) -> float:
    """Device time of one call in us.  The candidate is captured in a small CUDA graph (reps calls per replay) so that
    Python / launch overhead — which the training step does not pay either, it is a graph replay — stays out of the number."""
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    graph = None
    try:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            fn()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for _ in range(reps):
                fn()
    except Exception:  # noqa: BLE001  (an op that cannot be captured: fall back to eager timing)
        graph = None
        torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if graph is not None:
            graph.replay()
        else:
            for _ in range(reps):
                fn()
        e1.record(); e1.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3 / reps)
    ts.sort()
    return ts[len(ts) // 2]


# ---- the individual passes ---------------------------------------------------------------------------------------------
def _fprop_tc(x, w, stride, pad, stats, two_cta=False, impl=None):
    if impl in _HALO_KW:
        return _gemm.conv3x3_halo(x, w, False, stats=stats, **_HALO_KW[impl])
    if w.shape[2] == 1 and stride == 1:
        n, cin, h, wd = x.shape
        cout = w.shape[0]
        y2 = _gemm.gemm_tn(x.permute(0, 2, 3, 1).reshape(n * h * wd, cin), w.permute(0, 2, 3, 1).reshape(cout, cin), stats=stats, two_cta=two_cta)
        return y2.view(n, h, wd, cout).permute(0, 3, 1, 2)
    return _gemm.conv_fprop_nhwc(x, w, stride, pad, stats=stats, two_cta=two_cta)


def _dgrad_tc(dy, x, w, stride, pad, two_cta=False, impl=None):
    if impl in _HALO_KW:
        return _gemm.conv3x3_halo(dy, w, True, **_HALO_KW[impl])
    if w.shape[2] == 1 and stride == 2:
        return _gemm.conv1x1_s2_dgrad(dy, w)
    if w.shape[2] == 1 and stride == 1:
        n, cin, h, wd = x.shape
        cout = w.shape[0]
        dy2 = dy.permute(0, 2, 3, 1).reshape(n * h * wd, cout)
        return _gemm.gemm_nn(dy2, w.permute(0, 2, 3, 1).reshape(cout, cin), two_cta=two_cta).view(n, h, wd, cin).permute(0, 3, 1, 2)
    return _gemm.conv_dgrad_nhwc(dy, w, pad, two_cta=two_cta)


def _two_cta_caps(x, w, stride) -> dict:
    """CTA-pair variants: M (pixels) multiple of 256, output channels multiple of 128."""
    n, cin, h, wd = x.shape
    cout, _, k, _ = w.shape
    pad = k // 2
    p, q = (h + 2 * pad - k) // stride + 1, (wd + 2 * pad - k) // stride + 1
    m_ok = (n * p * q) % 256 == 0
    return {"fprop": m_ok and cout % 128 == 0, "dgrad": m_ok and cin % 128 == 0 and stride == 1}


def _halo_caps(x, w, stride) -> dict:
    """Halo-load kernels: 3x3, stride 1, whole image rows per 128-row tile (ops.gemm.halo_ok)."""
    off = {"fprop": False, "fprop2": False, "dgrad": False, "dgrad2": False}
    if not _HALO_STATE["enabled"] or not (x.is_cuda and x.dtype == torch.bfloat16):
        return off
    n, cin, h, wd = x.shape
    cout, _, k, _ = w.shape
    a = (n, h, wd)
    pair = os.environ.get("SHIPYARD_HALO_PAIR", "1") != "0"
    return {"fprop": _gemm.halo_ok(*a, cin, cout, k, k, stride, k // 2),
            "fprop2": pair and _gemm.halo_ok(*a, cin, cout, k, k, stride, k // 2, pair=True),
            "dgrad": _gemm.halo_ok(*a, cout, cin, k, k, stride, k // 2, dgrad=True),
            "dgrad2": pair and _gemm.halo_ok(*a, cout, cin, k, k, stride, k // 2, pair=True, dgrad=True)}


def experimental_impls(n: int, cin: int, h: int, wd: int, cout: int, k: int, stride: int) -> dict:
    """Not-yet-validated kernel variants that apply to a layer shape, per pass (pure function of the shape: testable on CPU).
    fprop / dgrad values are keys of ``_HALO_KW``; wgrad "th" is the halo-load wgrad kernel."""
    out = {"fprop": [], "dgrad": [], "wgrad": []}
    if (k, stride) != (3, 1) or cin % 64 or cout % 64:
        return out
    rows = _gemm.halo_rows(h, wd)
    if rows == 0:
        return out
    even_tiles = (n * (h // rows)) % 2 == 0
    small_box = (rows + 2) * (wd + 2) <= 184                 # fits the 23 KB halo slots of the weights-stationary pair kernel
    if cout == 64:                                           # BN = 64 tiles: one epilogue chunk per tile
        out["fprop"].append("tha")
        if even_tiles:
            out["fprop"] += ["th264", "th264a"]
    if cin == 64:                                            # dgrad writes cin channels
        out["dgrad"].append("tha")
    if cin == 128 and cout == 128 and even_tiles and small_box:
        out["fprop"].append("th2w")
        out["dgrad"].append("th2w")
    out["wgrad"].append("th")
    if _EXP_ALLOW is not None:
        out = {"fprop": [v for v in out["fprop"] if v in _EXP_ALLOW], "dgrad": [v for v in out["dgrad"] if v in _EXP_ALLOW],
               "wgrad": [v for v in out["wgrad"] if "wgrad_" + v in _EXP_ALLOW]}
    return out


def _close(a: torch.Tensor, ref: torch.Tensor) -> bool:
    a, ref = a.float(), ref.float()
    return bool(torch.isfinite(a).all()) and float((a - ref).abs().max()) <= 0.02 * float(ref.abs().max()) + 1e-3


def _halo_check(tag: str, key, got: torch.Tensor, ref: torch.Tensor) -> bool:
    """A halo candidate only enters the race if it reproduces the library result on this very call."""
    _HALO_STATE["checked"] += 1
    if _close(got, ref):
        return True
    _HALO_STATE["failed"].append(f"{tag}:{'x'.join(map(str, key))}")
    _HALO_STATE["enabled"] = False              # one wrong answer: stop using the kernels in this process
    return False


def _wgrad_tc(dy, x, w, stride, pad, out_view, accumulate, impl=None):
    """out_view: KRSC-dense [Cout,R,S,Cin] destination (the parameter's flat .grad) or None."""
    cout, cin, k, _ = w.shape
    if impl == "th":                                         # halo-load wgrad (experimental)
        if out_view is not None:
            _gemm.conv3x3_wgrad_halo(x, dy, out=out_view, accumulate=accumulate)
            return None
        return _gemm.conv3x3_wgrad_halo(x, dy)
    if k == 1 and stride == 1:
        n, _, h, wd = x.shape
        x2 = x.permute(0, 2, 3, 1).reshape(n * h * wd, cin)
        dy2 = dy.permute(0, 2, 3, 1).reshape(n * h * wd, cout)
        if out_view is not None:
            _gemm.gemm_nt_wgrad(x2, dy2, out=out_view.reshape(cout, cin), accumulate=accumulate)
            return None
        return _gemm.gemm_nt_wgrad(x2, dy2).view(cout, 1, 1, cin).permute(0, 3, 1, 2)
    if out_view is not None:
        _gemm.conv_wgrad_nhwc(x, dy, w.shape, stride, pad, out=out_view, accumulate=accumulate)
        return None
    return _gemm.conv_wgrad_nhwc(x, dy, w.shape, stride, pad)


def _cudnn_bwd(dy, x, w, stride, pad, want_dx, want_dw):
    dx, dw, _ = torch.ops.aten.convolution_backward(dy, x, w, None, [stride, stride], [pad, pad], [1, 1], False, [0, 0], 1,
                                                    [want_dx, want_dw, False])
    return dx, dw


def _grad_view(p: torch.Tensor) -> Optional[torch.Tensor]:
    g = getattr(p, "grad", None)
    if g is None or g.dtype != torch.bfloat16 or g.dim() != 4:
        return None
    v = g.permute(0, 2, 3, 1)
    return v if v.is_contiguous() else None


# ---- plan selection ------------------------------------------------------------------------------------------------------
def _autotune(x: torch.Tensor, w: torch.Tensor, stride: int) -> ConvPlan:
    caps = _tc_caps(x, w, stride)
    cout, cin, k, _ = w.shape
    pad = k // 2
    plan = ConvPlan(timings_us={})
    if _MODE == "cudnn" or not any(caps.values()):
        return plan
    hc = _halo_caps(x, w, stride)
    if _MODE == "tc":
        c2 = _two_cta_caps(x, w, stride)
        fp = ("tc2" if c2["fprop"] else "tc") if caps["fprop"] else "cudnn"
        dg = ("tc2" if c2["dgrad"] else "tc") if caps["dgrad"] else "cudnn"
        # forced mode: the halo kernels where they measured faster than the im2col ones (profiles/conv_halo.md): rows of >= 28 pixels
        if hc["fprop"] and x.shape[3] >= 28:
            fp = "th2" if hc["fprop2"] else "th"
        if hc["dgrad"] and x.shape[3] >= 28:
            dg = "th2" if hc["dgrad2"] else "th"
        return ConvPlan(fp, dg, "tc" if caps["wgrad"] else "cudnn",
                        stats=caps["fprop"] and (k > 1 or stride > 1 or cin >= 256), timings_us={})
    t = plan.timings_us
    with torch.no_grad():
        xd, wd_ = x.detach(), w.detach()
        y = F.conv2d(xd, wd_, None, stride, pad)
        t_stats_pass = y.numel() * 2 / _HBM_BPS * 1e6 + 3.0            # the separate statistics kernel a non-fused fprop needs
        t["fprop_cudnn"] = _time(lambda: F.conv2d(xd, wd_, None, stride, pad)) + t_stats_pass
        caps2 = _two_cta_caps(x, w, stride)
        if caps["fprop"]:
            st = torch.zeros(2 * cout, dtype=torch.float32, device=x.device)
            t["fprop_tc_stats"] = _time(lambda: _fprop_tc(xd, wd_, stride, pad, st))
            t["fprop_tc"] = _time(lambda: _fprop_tc(xd, wd_, stride, pad, None)) + t_stats_pass
            cands = ["fprop_cudnn", "fprop_tc_stats", "fprop_tc"]
            if caps2["fprop"]:
                t["fprop_tc2_stats"] = _time(lambda: _fprop_tc(xd, wd_, stride, pad, st, True))
                t["fprop_tc2"] = _time(lambda: _fprop_tc(xd, wd_, stride, pad, None, True)) + t_stats_pass
                cands += ["fprop_tc2_stats", "fprop_tc2"]
            for impl, cap in (("th", "fprop"), ("th2", "fprop2")):
                if hc[cap] and _HALO_STATE["enabled"] and _halo_check("fprop_" + impl, _key(x, w, stride), _fprop_tc(xd, wd_, stride, pad, None, impl=impl), y):
                    t[f"fprop_{impl}_stats"] = _time(lambda: _fprop_tc(xd, wd_, stride, pad, st, impl=impl))
                    t[f"fprop_{impl}"] = _time(lambda: _fprop_tc(xd, wd_, stride, pad, None, impl=impl)) + t_stats_pass
                    cands += [f"fprop_{impl}_stats", f"fprop_{impl}"]
            exp = experimental_impls(*_key(x, w, stride)[:4], cout, k, stride) if (_EXP and _HALO_STATE["enabled"]) else {"fprop": [], "dgrad": [], "wgrad": []}
            for impl in exp["fprop"]:
                if _HALO_STATE["enabled"] and _halo_check("fprop_" + impl, _key(x, w, stride), _fprop_tc(xd, wd_, stride, pad, None, impl=impl), y):
                    t[f"fprop_{impl}_stats"] = _time(lambda: _fprop_tc(xd, wd_, stride, pad, st, impl=impl))
                    t[f"fprop_{impl}"] = _time(lambda: _fprop_tc(xd, wd_, stride, pad, None, impl=impl)) + t_stats_pass
                    cands += [f"fprop_{impl}_stats", f"fprop_{impl}"]
            best = _pick({k_: t[k_] for k_ in cands}, "fprop_")
            plan.fprop = best.split("_")[1]
            plan.stats = best.endswith("_stats")
        dy = torch.randn_like(y).contiguous(memory_format=torch.channels_last)
        t["dgrad_cudnn"] = _time(lambda: _cudnn_bwd(dy, xd, wd_, stride, pad, True, False))
        if caps["dgrad"]:
            t["dgrad_tc"] = _time(lambda: _dgrad_tc(dy, xd, wd_, stride, pad))
            if caps2["dgrad"]:
                t["dgrad_tc2"] = _time(lambda: _dgrad_tc(dy, xd, wd_, stride, pad, True))
            if hc["dgrad"] and _HALO_STATE["enabled"]:
                dx_ref = _cudnn_bwd(dy, xd, wd_, stride, pad, True, False)[0]
                for impl, cap in (("th", "dgrad"), ("th2", "dgrad2")):
                    if hc[cap] and _HALO_STATE["enabled"] and _halo_check("dgrad_" + impl, _key(x, w, stride), _dgrad_tc(dy, xd, wd_, stride, pad, impl=impl), dx_ref):
                        t[f"dgrad_{impl}"] = _time(lambda: _dgrad_tc(dy, xd, wd_, stride, pad, impl=impl))
            if _EXP and _HALO_STATE["enabled"]:
                exp_d = experimental_impls(*_key(x, w, stride)[:4], cout, k, stride)["dgrad"]
                if exp_d:
                    dx_ref = _cudnn_bwd(dy, xd, wd_, stride, pad, True, False)[0]
                for impl in exp_d:
                    if _HALO_STATE["enabled"] and _halo_check("dgrad_" + impl, _key(x, w, stride), _dgrad_tc(dy, xd, wd_, stride, pad, impl=impl), dx_ref):
                        t[f"dgrad_{impl}"] = _time(lambda: _dgrad_tc(dy, xd, wd_, stride, pad, impl=impl))
            plan.dgrad = _pick(t, "dgrad_").split("_")[1]
        t_accum = w.numel() * 6 / 4e12 * 1e6 + 3.0                     # AccumulateGrad add the library path pays
        t["wgrad_cudnn"] = _time(lambda: _cudnn_bwd(dy, xd, wd_, stride, pad, False, True)) + t_accum
        if caps["wgrad"]:
            buf = torch.zeros((cout, k, k, cin), dtype=torch.bfloat16, device=x.device)
            t["wgrad_tc"] = _time(lambda: _wgrad_tc(dy, xd, wd_, stride, pad, buf, True))
            if _EXP and _HALO_STATE["enabled"] and "th" in experimental_impls(*_key(x, w, stride)[:4], cout, k, stride)["wgrad"]:
                dw_ref = _cudnn_bwd(dy, xd, wd_, stride, pad, False, True)[1]
                if _halo_check("wgrad_th", _key(x, w, stride), _wgrad_tc(dy, xd, wd_, stride, pad, None, False, impl="th"), dw_ref):
                    buf.zero_()
                    t["wgrad_th"] = _time(lambda: _wgrad_tc(dy, xd, wd_, stride, pad, buf, True, impl="th"))
            plan.wgrad = _pick(t, "wgrad_").split("_")[1]
    plan.timings_us = {k_: round(v, 1) for k_, v in t.items()}
    return plan


def plan_for(x: torch.Tensor, w: torch.Tensor, stride: int) -> ConvPlan:
    key = _key(x, w, stride)
    p = _PLANS.get(key)
    if p is None:
        if not (x.is_cuda and x.dtype == torch.bfloat16) or torch.cuda.is_current_stream_capturing():
            return ConvPlan()                      # never measure inside a graph capture; the warm-up step has filled the table
        p = _PLANS[key] = _autotune(x, w, stride)
    return p


class _Conv(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w, stride, plan: ConvPlan):
        ctx.set_materialize_grads(False)          # the statistics output has no gradient: do not let autograd build a zeros tensor for it
        k = w.shape[2]
        pad = k // 2
        stats = None
        if plan.fprop != "cudnn":
            if plan.stats:
                stats = _fused_zeros(2 * w.shape[0], x.device)          # slice of the step's zero pool (one memset per step)
            y = _fprop_tc(x, w, stride, pad, stats, plan.fprop == "tc2", impl=plan.fprop)
        else:
            y = F.conv2d(x, w, None, stride, pad)
        ctx.save_for_backward(x, w)
        ctx.stride, ctx.pad, ctx.plan, ctx.w_ref = stride, pad, plan, w
        if stats is not None:
            ctx.mark_non_differentiable(stats)
        return y, stats

    @staticmethod
    def backward(ctx, dy, _ds):
        x, w = ctx.saved_tensors
        plan, stride, pad = ctx.plan, ctx.stride, ctx.pad
        if not dy.is_contiguous(memory_format=torch.channels_last):
            dy = dy.contiguous(memory_format=torch.channels_last)
        dx = dw = None
        need_dx, need_dw = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        lib_dx = need_dx and plan.dgrad == "cudnn"
        lib_dw = need_dw and plan.wgrad == "cudnn"
        if lib_dx or lib_dw:
            dx, dw = _cudnn_bwd(dy, x, w, stride, pad, lib_dx, lib_dw)
        if need_dx and plan.dgrad != "cudnn":
            dx = _dgrad_tc(dy, x, w, stride, pad, plan.dgrad == "tc2", impl=plan.dgrad)
        if need_dw and plan.wgrad != "cudnn":
            dw = _wgrad_tc(dy, x, w, stride, pad, _grad_view(ctx.w_ref), True,      # None when written into .grad in place
                           impl=plan.wgrad if plan.wgrad != "tc" else None)
        return dx, dw, None, None


# ---- inference: convolution + folded BatchNorm (+ residual) (+ ReLU) ------------------------------------------------------------------
# A table of its own, so the training plans (and bench.py's report of them) never change because an evaluation ran.  Two candidates
# per shape: the own tcgen05 kernel with the affine epilogue (ops.gemm.conv_affine_nhwc), and cuDNN followed by ops.fused.bn_infer_apply.
_INFER_PLANS: dict = {}


@dataclass
class InferPlan:
    impl: str = "cudnn"       # "tc" (conv_affine_nhwc) | "cudnn" (F.conv2d + bn_infer_apply)
    timings_us: Optional[dict] = None


def infer_plan_table() -> dict:
    return {"x".join(map(str, k)): asdict(v) for k, v in _INFER_PLANS.items()}


def _infer_key(x, w, stride, residual, relu):
    return _key(x, w, stride) + (int(residual), int(relu))


def _infer_tc(x, w, scale, shift, stride, residual, relu):
    return _gemm.conv_affine_nhwc(x, w, scale, shift, stride, residual=residual, relu=relu)


def _infer_cudnn(x, w, scale, shift, stride, residual, relu):
    from .fused import bn_infer_apply
    y = F.conv2d(x, w, None, stride, w.shape[2] // 2)
    if not y.is_contiguous(memory_format=torch.channels_last):
        y = y.contiguous(memory_format=torch.channels_last)
    return bn_infer_apply(y, scale, shift, residual, relu, out=y)


def infer_plan_for(x: torch.Tensor, w: torch.Tensor, stride: int, residual: bool, relu: bool, use_tc: bool = True) -> InferPlan:
    """The inference implementation of one layer shape: raced once (device-timed, outside any graph capture) in ``auto`` mode,
    the own kernel wherever it applies in ``tc`` mode, cuDNN in ``cudnn`` mode or when ``use_tc`` (the layer's use_tc_gemm) is off."""
    key = _infer_key(x, w, stride, residual, relu)
    p = _INFER_PLANS.get(key)
    if p is not None:
        return p
    ok = use_tc and _gemm.conv_affine_ok(x, w, stride)
    if _MODE == "cudnn" or not ok:
        p = InferPlan("cudnn", {})
    elif _MODE == "tc":
        p = InferPlan("tc", {})
    else:
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError("infer_plan_for: shape %s was not raced before graph capture" % (key,))
        cout = w.shape[0]
        scale = torch.rand(cout, device=x.device) + 0.5
        shift = torch.randn(cout, device=x.device)
        n, _, h, wd = x.shape
        k = w.shape[2]
        pq = ((h + 2 * (k // 2) - k) // stride + 1, (wd + 2 * (k // 2) - k) // stride + 1)
        r = torch.randn((n, cout) + pq, device=x.device).to(torch.bfloat16).contiguous(memory_format=torch.channels_last) if residual else None
        xd, wd_ = x.detach(), w.detach()
        with torch.no_grad():
            t = {"fprop_cudnn": _time(lambda: _infer_cudnn(xd, wd_, scale, shift, stride, r, relu)),
                 "fprop_tc": _time(lambda: _infer_tc(xd, wd_, scale, shift, stride, r, relu))}
        p = InferPlan(_pick(t, "fprop_").split("_")[1], {k_: round(v, 1) for k_, v in t.items()})
    _INFER_PLANS[key] = p
    return p


def conv_bn_infer(x: torch.Tensor, w: torch.Tensor, scale: torch.Tensor, shift: torch.Tensor, stride: int = 1,
                  residual: Optional[torch.Tensor] = None, relu: bool = True, use_tc: bool = True) -> torch.Tensor:
    """act(conv2d(x, w) * scale + shift (+ residual)) through the layer shape's inference plan (channels_last bf16)."""
    plan = infer_plan_for(x, w, stride, residual is not None, relu, use_tc)
    fn = _infer_tc if plan.impl == "tc" else _infer_cudnn
    return fn(x, w, scale, shift, stride, residual, relu)


def conv_bn_input(x: torch.Tensor, w: torch.Tensor, stride: int = 1):
    """Convolution (kernel 1 or 3, 'same' padding) for a following BatchNorm: returns (y, stats or None)."""
    return _Conv.apply(x, w, stride, plan_for(x, w, stride))
