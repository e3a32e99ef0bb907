"""Inference on the sm_100a kernels: the folded-BN epilogue of the tcgen05 GEMM / im2col convolution, bn_infer_apply, the index-free
max-pool, the graph-captured ResNet engine against torchvision (calibrated bf16 noise floor, every dispatcher mode), evaluate() between
captured training steps, evaluate() at world 2, and the scoring recipe end to end."""
import json
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

from _mp import run_ranks

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():
    pytest.skip("needs a GPU", allow_module_level=True)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NOISE_FACTOR = 2.0
ABS_SLACK = 0.01


def _resnet50_conv_shapes(n=32):
    """(n, cin, h, w, cout, k, stride) of every distinct convolution of ResNet-50 after the stem (224 x 224 input)."""
    from batch_shipyard_b200.models.resnet import resnet50
    m = resnet50()
    shapes, h = [], 56
    for b in m.blocks:
        s = b.c2.stride
        for c, hh in ((b.c1, h), (b.c2, h), (b.c3, h // s)) + (((b.down, h),) if b.down is not None else ()):
            shapes.append((n, c.cin, hh, hh, c.cout, c.k, c.stride))
        h //= s
    return sorted(set(shapes))


def _case(n, cin, h, w, cout, k, stride, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(n, cin, h, w, device="cuda", generator=g).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    wt = (torch.randn(cout, cin, k, k, device="cuda", generator=g) * 0.25).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    p = (h + 2 * (k // 2) - k) // stride + 1
    q = (w + 2 * (k // 2) - k) // stride + 1
    scale = torch.rand(cout, device="cuda", generator=g) + 0.5
    shift = torch.randn(cout, device="cuda", generator=g)
    res = torch.randn(n, cout, p, q, device="cuda", generator=g).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    return x, wt, scale, shift, res


SHAPES = _resnet50_conv_shapes() + [(7, 64, 11, 13, 128, 1, 1),      # ragged M: 1001 rows (GEMM path)
                                    (4, 128, 16, 16, 72, 1, 1),      # N = 72
                                    (2, 64, 16, 16, 72, 3, 1)]       # N = 72 on the im2col kernel


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_affine_epilogue_matches_fp32_reference(shape):
    from batch_shipyard_b200.ops import gemm
    n, cin, h, w, cout, k, stride = shape
    x, wt, scale, shift, res = _case(*shape)
    if not gemm.conv_affine_ok(x, wt, stride):
        pytest.skip("shape outside the own kernel's constraints (N*P*Q % 128): cuDNN + bn_infer_apply serve it")
    conv = F.conv2d(x.float(), wt.float(), None, stride, k // 2)
    kdim = cin * k * k
    for relu in (False, True):
        for r in (None, res):
            ref = conv * scale.view(1, -1, 1, 1) + shift.view(1, -1, 1, 1)
            if r is not None:
                ref = ref + r.float()
            if relu:
                ref = torch.relu(ref)
            got = gemm.conv_affine_nhwc(x, wt, scale, shift, stride, residual=r, relu=relu)
            assert got.is_contiguous(memory_format=torch.channels_last)
            torch.testing.assert_close(got.float(), ref, atol=0.02 * (kdim ** 0.5) * 0.25 * 1.5 + 0.05, rtol=2e-2)


@pytest.mark.parametrize("shape", [s for s in SHAPES if s[5] == 1 and s[6] == 1][:4] + [s for s in SHAPES if s[5] == 3][:3],
                         ids=lambda s: "x".join(map(str, s)))
def test_affine_epilogue_identity_is_bit_identical_to_plain_kernels(shape):
    from batch_shipyard_b200.ops import gemm
    n, cin, h, w, cout, k, stride = shape
    x, wt, _, _, _ = _case(*shape, seed=3)
    if not gemm.conv_affine_ok(x, wt, stride):
        pytest.skip("outside the own kernel's constraints")
    one, zero = torch.ones(cout, device="cuda"), torch.zeros(cout, device="cuda")
    got = gemm.conv_affine_nhwc(x, wt, one, zero, stride, residual=None, relu=False)
    if k == 1 and stride == 1:
        plain = gemm.gemm_tn(x.permute(0, 2, 3, 1).reshape(-1, cin), wt.permute(0, 2, 3, 1).reshape(cout, cin))
        assert torch.equal(got.permute(0, 2, 3, 1).reshape(-1, cout), plain)
    else:
        assert torch.equal(got, gemm.conv_fprop_nhwc(x, wt, stride, k // 2))


def test_affine_rejects_output_aliasing_residual():
    from batch_shipyard_b200.ops import gemm
    import ctypes as C
    x, wt, scale, shift, res = _case(2, 64, 8, 8, 64, 1, 1)
    lib = gemm.load()
    buf = res.permute(0, 2, 3, 1)
    rc = lib.sy_gemm_bf16_tn_affine(C.c_void_p(x.data_ptr()), C.c_void_p(wt.data_ptr()), C.c_void_p(buf.data_ptr()), 128, 64, 64, 64, 64, 64,
                                    C.c_void_p(scale.data_ptr()), C.c_void_p(shift.data_ptr()), C.c_void_p(buf.data_ptr()), 64, 1, 0, 0,
                                    C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc != 0 and b"alias" in lib.sy_gemm_last_error()


def test_bn_infer_apply_and_fold_match_torch():
    from batch_shipyard_b200.ops import fused
    g = torch.Generator(device="cuda").manual_seed(5)
    c = 96
    x = torch.randn(3, c, 9, 7, device="cuda", generator=g).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    r = torch.randn(3, c, 9, 7, device="cuda", generator=g).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    gamma = (torch.rand(c, device="cuda", generator=g) + 0.5).to(torch.bfloat16)
    beta = torch.randn(c, device="cuda", generator=g).to(torch.bfloat16)
    mean = torch.randn(c, device="cuda", generator=g)
    var = torch.rand(c, device="cuda", generator=g) + 0.1
    tab = fused.BnFoldTable([(gamma, beta, mean, var, 1e-5), (gamma[:64].contiguous(), beta[:64].contiguous(), mean[:64].contiguous(),
                                                              var[:64].contiguous(), 1e-3)], "cuda")
    fused.bn_fold(tab)
    for i, eps in ((0, 1e-5), (1, 1e-3)):
        cc = tab.scale[i].numel()
        s_ref, t_ref = fused.bn_fold_reference(gamma[:cc], beta[:cc], mean[:cc], var[:cc], eps)
        torch.testing.assert_close(tab.scale[i], s_ref, rtol=1e-6, atol=1e-6)
        torch.testing.assert_close(tab.shift[i], t_ref, rtol=1e-6, atol=1e-6)
    s, t = tab.scale[0], tab.shift[0]
    for relu in (False, True):
        for res in (None, r):
            ref = x.float() * s.view(1, -1, 1, 1) + t.view(1, -1, 1, 1) + (0 if res is None else res.float())
            ref = torch.relu(ref) if relu else ref
            got = fused.bn_infer_apply(x, s, t, res, relu)
            torch.testing.assert_close(got.float(), ref.to(torch.bfloat16).float(), atol=1e-5, rtol=1e-2)
            ev = F.batch_norm(x.float(), mean, var, gamma.float(), beta.float(), training=False, eps=1e-5)
            ev = ev + (0 if res is None else res.float())
            torch.testing.assert_close(got.float(), torch.relu(ev) if relu else ev, atol=3e-2, rtol=2e-2)


def test_index_free_maxpool_matches_exactly():
    from batch_shipyard_b200.ops import fused
    x = torch.randn(4, 64, 56, 56, device="cuda").to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    got = fused.maxpool3x3s2_infer(x)
    assert torch.equal(got, F.max_pool2d(x.float(), 3, 2, 1).to(torch.bfloat16))
    assert torch.equal(got, fused.maxpool3x3s2(x))


# ---- whole model --------------------------------------------------------------------------------------------------------------
def _random_tv(seed=0):
    torchvision = pytest.importorskip("torchvision")
    torch.manual_seed(seed)
    tv = torchvision.models.resnet50()
    with torch.no_grad():
        for m in tv.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.weight.uniform_(0.5, 1.5); m.bias.uniform_(-0.3, 0.3)
                m.running_mean.uniform_(-0.2, 0.2); m.running_var.uniform_(0.5, 2.0)
    return tv.eval()


def _images(n, size=224, seed=7):
    from batch_shipyard_b200.ops import fused
    g = torch.Generator(device="cuda").manual_seed(seed)
    img = torch.randint(0, 256, (n, size, size, 3), dtype=torch.uint8, device="cuda", generator=g)
    mean = torch.tensor(fused.IMAGENET_MEAN, device="cuda"); std = torch.tensor(fused.IMAGENET_STD, device="cuda")
    return img, ((img.float() / 255.0 - mean) / std).permute(0, 3, 1, 2).contiguous()


def _rel(a, b):
    return float((a.float() - b.float()).norm() / b.float().norm().clamp_min(1e-12))


def _floor(module, x_ref, ref):
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        lo = module.to(memory_format=torch.channels_last)(x_ref.contiguous(memory_format=torch.channels_last)).float()
    return _rel(lo, ref)


@pytest.mark.parametrize("mode", ["auto", "tc", "cudnn"])
def test_engine_resnet50_matches_torchvision_fp32(mode):
    from batch_shipyard_b200.models.resnet import load_torchvision_state_dict, resnet50
    from batch_shipyard_b200.ops import conv
    from batch_shipyard_b200.parallel.infer import ResNetInference, cast_for_inference
    tv = _random_tv().cuda()
    ours = resnet50()
    load_torchvision_state_dict(ours, tv.state_dict())
    cast_for_inference(ours, "cuda")
    img, x_ref = _images(16)
    with torch.no_grad():
        ref = tv(x_ref).float()
    floor = _floor(tv, x_ref, ref)
    conv.set_mode(mode)
    try:
        eng = ResNetInference(ours, 16)
        got = eng(img)
        table = conv.infer_plan_table()
    finally:
        conv.set_mode("auto")
    rel = _rel(got, ref)
    own = sum(1 for v in table.values() if v["impl"] == "tc")
    print(f"[{mode}] engine rel {rel:.4f} floor {floor:.4f} own-kernel shapes {own}/{len(table)} kernels/batch {eng.kernels_per_batch}")
    assert got.dtype == torch.float32 and tuple(got.shape) == (16, 1000)
    assert rel <= NOISE_FACTOR * floor + ABS_SLACK, (mode, rel, floor)
    if mode == "tc":
        assert own > 0
    if mode == "cudnn":
        assert own == 0
    # a short final batch is zero-padded and sliced: the first rows are unchanged
    torch.testing.assert_close(eng(img[:5]), got[:5], rtol=0, atol=0)


@pytest.mark.parametrize("name", ["resnet_tiny", "resnet20_cifar"])
def test_engine_small_models_match_their_own_fp32_eval(name):
    from batch_shipyard_b200.models import resnet
    from batch_shipyard_b200.ops import fused
    from batch_shipyard_b200.parallel.infer import ResNetInference, cast_for_inference
    torch.manual_seed(1)
    m = getattr(resnet, name)(10)
    with torch.no_grad():
        for mod in m.modules():
            if isinstance(mod, resnet.ConvBN):
                mod.gamma.uniform_(0.5, 1.5); mod.beta.uniform_(-0.3, 0.3)
                mod.running_mean.uniform_(-0.2, 0.2); mod.running_var.uniform_(0.5, 2.0)
    ref_m = getattr(resnet, name)(10)
    ref_m.load_state_dict(m.state_dict())
    ref_m = ref_m.cuda().eval()
    size = 32 if name == "resnet20_cifar" else 64
    img, _ = _images(8, size)
    if name == "resnet_tiny":                       # the trainer's conversion: space-to-depth stem input
        xs = torch.empty(8, size // 2 + 3, size // 2 + 3, 16, dtype=torch.bfloat16, device="cuda")
        fused.u8_to_s2d_norm(img, xs)
    else:
        xs = torch.empty(8, size, size, 3, dtype=torch.bfloat16, device="cuda")
        fused.u8_to_bf16_norm(img, xs)
    x_ref = xs.float().permute(0, 3, 1, 2).contiguous()
    with torch.no_grad():
        ref = ref_m(x_ref).float()
    floor = _floor(ref_m, x_ref, ref)
    eng = ResNetInference(cast_for_inference(m, "cuda"), 8, image_size=size)
    rel = _rel(eng(img), ref)
    print(f"[{name}] engine rel {rel:.4f} floor {floor:.4f}")
    assert rel <= NOISE_FACTOR * floor + ABS_SLACK, (name, rel, floor)


def test_graph_replay_equals_eager_call_and_plan_table_lists_every_shape():
    from batch_shipyard_b200.models.resnet import resnet50
    from batch_shipyard_b200.ops import conv
    from batch_shipyard_b200.parallel.infer import ResNetInference, cast_for_inference
    torch.manual_seed(0)
    m = cast_for_inference(resnet50(), "cuda")
    eng = ResNetInference(m, 8)
    img, _ = _images(8, seed=11)
    g = eng(img)
    with torch.no_grad():
        eng._forward()                               # the same call, eager
    torch.cuda.synchronize()
    assert torch.equal(eng.static_logits, g)
    table = conv.infer_plan_table()
    want = set()
    h = 56
    for b in m.blocks:
        s = b.c2.stride
        for c, hh, res in ((b.c1, h, False), (b.c2, h, False), (b.c3, h // s, True)) + (((b.down, h, False),) if b.down is not None else ()):
            want.add("x".join(map(str, (8, c.cin, hh, hh, c.cout, c.k, c.stride, int(res), int(c.relu)))))
        h //= s
    assert want <= set(table), sorted(want - set(table))
    assert eng.kernels_per_batch > 0


def test_evaluate_between_captured_steps_leaves_training_state_bitwise():
    from batch_shipyard_b200.models.resnet import resnet_tiny
    from batch_shipyard_b200.ops.coll import Communicator
    from batch_shipyard_b200.parallel.ddp import FusedDataParallelTrainer
    torch.manual_seed(0)
    comm = Communicator(0, 1, device=0, heap_bytes=256 << 20)
    tr = FusedDataParallelTrainer(resnet_tiny(10), comm, (16, 3, 64, 64), 10, lr=0.05)
    img, _ = _images(16, 64, seed=1)
    y = torch.randint(0, 10, (16,), device="cuda")
    tr.load_images_u8(img, y)
    tr.prepare(warmup=1)
    for _ in range(2):
        tr.step()
    torch.cuda.synchronize()
    snap = {"params": tr.flat.params, "grads": tr.flat.grads, "master": tr.flat.master, "momentum": tr.flat.momentum,
            "static_x": tr.static_x, "static_y": tr.static_y, "static_loss": tr.static_loss}
    snap.update({"buf." + k: v for k, v in tr.model.named_buffers()})
    snap = {k: v.detach().clone() for k, v in snap.items()}
    graph, training = tr.graph, tr.model.training
    ev_img, _ = _images(40, 64, seed=2)
    ev = tr.evaluate(ev_img, torch.randint(0, 10, (40,), device="cuda"), batch=16)
    torch.cuda.synchronize()
    assert ev["count"] == 40 and 0 <= ev["top1"] <= ev["top5"] <= 40
    now = {"params": tr.flat.params, "grads": tr.flat.grads, "master": tr.flat.master, "momentum": tr.flat.momentum,
           "static_x": tr.static_x, "static_y": tr.static_y, "static_loss": tr.static_loss}
    now.update({"buf." + k: v for k, v in tr.model.named_buffers()})
    for k, v in snap.items():
        assert torch.equal(now[k], v), k
    assert tr.graph is graph and tr.model.training == training
    loss = float(tr.step())
    assert loss == loss and abs(loss) < 100
    comm.close()


@pytest.mark.multigpu
def test_evaluate_world2_sums_the_per_rank_references(tmp_path):
    ok, outs = run_ranks("_infer_worker.py", 2, extra=["--out", str(tmp_path), "--image", "64"], gpu=True, timeout=600)
    assert ok, "\n".join(outs)
    evs = [json.loads(next(l for l in o.splitlines() if l.startswith("EVAL "))[5:]) for o in outs]
    refs = [json.load(open(tmp_path / f"ref.rank{r}.json")) for r in range(2)]
    assert evs[0] == evs[1] and evs[0]["count"] == sum(r["count"] for r in refs)
    # bf16 engine against an fp32 reference: hits may differ on near-ties, never by much
    assert abs(evs[0]["top5"] - sum(r["top5"] for r in refs)) <= 3


def test_score_recipe_with_torchvision_weights_agrees_with_fp32(tmp_path):
    import numpy as np
    tv = _random_tv(3).cuda()
    wpath = tmp_path / "w.pt"
    torch.save(tv.state_dict(), wpath)
    img, x_ref = _images(48, seed=21)
    np.save(tmp_path / "x.npy", img.cpu().numpy())
    env = dict(os.environ, RANK="0", WORLD_SIZE="1", SHIPYARD_GPU="0")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "recipes", "PyTorch-GPU", "score_resnet50.py"), "--images", str(tmp_path / "x.npy"),
                        "--weights", str(wpath), "--batch", "32", "--out", str(tmp_path / "out")], env=env, cwd=ROOT,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert p.returncode == 0, p.stdout[-3000:]
    out = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    assert out["images"] == 48 and out["own_kernels_per_batch"] > 0, out
    top5 = torch.from_numpy(np.load(tmp_path / "out" / "top5.rank0.npy")).cuda()
    with torch.no_grad():
        ref = tv(x_ref).float()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            lo = tv(x_ref).float()
    # per image, the noise floor of bf16 arithmetic on this network: stock bf16 autocast against fp32, largest error over the classes
    noise = (lo - ref).abs().max(dim=1).values
    margin = NOISE_FACTOR * noise + ABS_SLACK * ref.std(dim=1)
    srt = ref.sort(dim=1, descending=True)
    b5, b6 = srt.values[:, 4], srt.values[:, 5]                     # fp32 top-5 boundary: 5th and 6th largest logit
    # the check separates right from wrong: a class picked at random sits far below the boundary compared with the margin
    assert float((b5 - ref.median(dim=1).values).median()) > 4 * float(margin.median()), (b5, margin)
    picked = ref.gather(1, top5)                                    # fp32 logits of the engine's top-5 classes
    # every class the engine ranks in its top 5 is in the fp32 top 5 or within the noise floor of a tie with its boundary
    low = picked < (b5 - margin).view(-1, 1)
    assert not bool(low.any()), [(i, top5[i].tolist(), srt.indices[i, :5].tolist()) for i in torch.nonzero(low.any(dim=1)).flatten().tolist()]
    # every fp32 class that is clearly inside the top 5 (above the 6th by more than the noise floor) is in the engine's top 5
    for i in range(ref.shape[0]):
        clear = set(torch.nonzero(ref[i] > b6[i] + margin[i]).flatten().tolist())
        assert clear <= set(top5[i].tolist()), (i, sorted(clear), top5[i].tolist())
