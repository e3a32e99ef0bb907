"""Inference and evaluation without a GPU: the BatchNorm fold formula, torchvision weight import, FusedDataParallelTrainer.evaluate at
world 2 on the stub transport, the recipe bodies (train --eval-batches, batch scoring) and the scoring job variant."""
import json
import os
import subprocess
import sys
import uuid

import pytest
import torch
import torch.nn.functional as F

from _mp import run_ranks

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bn_fold_formula_equals_eval_batch_norm():
    from batch_shipyard_b200.ops.fused import bn_fold_reference
    g = torch.Generator().manual_seed(0)
    c = 96
    x = torch.randn(4, c, 5, 7, generator=g, dtype=torch.float64)
    gamma, beta = torch.rand(c, generator=g, dtype=torch.float64) + 0.5, torch.randn(c, generator=g, dtype=torch.float64)
    mean, var = torch.randn(c, generator=g, dtype=torch.float64), torch.rand(c, generator=g, dtype=torch.float64) * 3 + 0.01
    for eps in (1e-5, 1e-3):
        ref = F.batch_norm(x, mean, var, gamma, beta, training=False, eps=eps)
        scale, shift = bn_fold_reference(gamma.double(), beta.double(), mean, var, eps)
        # bn_fold_reference returns fp32 (the kernel's precision): compare at fp32 resolution
        got = x * scale.double().view(1, -1, 1, 1) + shift.double().view(1, -1, 1, 1)
        assert torch.allclose(got, ref, rtol=1e-6, atol=1e-6), float((got - ref).abs().max())


def _random_torchvision_resnet50(seed=0):
    torchvision = pytest.importorskip("torchvision")
    torch.manual_seed(seed)
    tv = torchvision.models.resnet50()
    with torch.no_grad():
        for m in tv.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.weight.uniform_(0.5, 1.5); m.bias.uniform_(-0.5, 0.5)
                m.running_mean.uniform_(-0.3, 0.3); m.running_var.uniform_(0.5, 2.0)
    return tv.eval()


def test_torchvision_import_round_trip_matches_torchvision_eval():
    from batch_shipyard_b200.models.resnet import load_torchvision_state_dict, resnet50
    tv = _random_torchvision_resnet50()
    ours = resnet50()
    load_torchvision_state_dict(ours, tv.state_dict())
    ours.eval()
    x = torch.randn(2, 3, 64, 64, generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        ref, got = tv(x), ours(x)
    rel = float((got - ref).norm() / ref.norm())
    assert rel < 1e-4, rel
    # the running statistics came along, num_batches_tracked was ignored
    assert torch.equal(ours.blocks[3].c2.running_var, tv.layer2[0].bn2.running_var)


def test_torchvision_import_rejects_unused_missing_and_misshaped_keys():
    from batch_shipyard_b200.models.resnet import load_torchvision_state_dict, resnet50
    tv = _random_torchvision_resnet50()
    sd = tv.state_dict()
    ours = resnet50()
    before = ours.fc_weight.detach().clone()
    bad = dict(sd); bad["layer5.0.conv1.weight"] = torch.zeros(1)
    with pytest.raises(KeyError, match="unused keys: layer5.0.conv1.weight"):
        load_torchvision_state_dict(ours, bad)
    bad = dict(sd); del bad["layer3.2.bn2.running_mean"]
    with pytest.raises(KeyError, match="missing keys: layer3.2.bn2.running_mean"):
        load_torchvision_state_dict(ours, bad)
    bad = dict(sd); bad["fc.weight"] = torch.zeros(10, 2048)
    with pytest.raises(KeyError, match=r"shape mismatch: fc.weight \(10, 2048\)"):
        load_torchvision_state_dict(ours, bad)
    assert torch.equal(ours.fc_weight, before)                   # a refused import changes nothing


def test_evaluate_world2_stub_sums_the_per_rank_references(tmp_path):
    ok, outs = run_ranks("_infer_worker.py", 2, extra=["--out", str(tmp_path)], gpu=False, timeout=300)
    assert ok, "\n".join(outs)
    evs = [json.loads(next(l for l in o.splitlines() if l.startswith("EVAL "))[5:]) for o in outs]
    refs = [json.load(open(tmp_path / f"ref.rank{r}.json")) for r in range(2)]
    assert evs[0] == evs[1]                                      # every rank gets the job-wide sums
    ev = evs[0]
    assert ev["count"] == sum(r["count"] for r in refs) == 20 + 24
    assert ev["top1"] == sum(r["top1"] for r in refs) and ev["top5"] == sum(r["top5"] for r in refs)
    assert abs(ev["loss"] - sum(r["loss"] for r in refs)) < 1e-3 * max(1.0, abs(ev["loss"]))


def _run_world(args, script, world=2, timeout=600):
    session = "inf" + uuid.uuid4().hex[:10]
    procs = [subprocess.Popen([sys.executable, os.path.join(ROOT, script)] + args, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                              cwd=ROOT, env=dict(os.environ, RANK=str(r), WORLD_SIZE=str(world), SHIPYARD_GPU="-1", SHIPYARD_COLL_SESSION=session,
                                                 OMP_NUM_THREADS="2"))
             for r in range(world)]
    outs = [p.communicate(timeout=timeout)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(outs)
    return json.loads([l for l in outs[0].splitlines() if l.startswith("{")][-1])


def test_train_recipe_eval_batches_world2():
    out = _run_world(["--model", "resnet20", "--steps", "3", "--batch", "16", "--eval-batches", "2"], "recipes/PyTorch-GPU/train_resnet50.py")
    ev = out["eval"]
    assert ev["count"] == 2 * 2 * 16 and 0 <= ev["top1"] <= ev["top5"] <= ev["count"] and ev["loss"] > 0, out
    assert "test_accuracy" in out                              # the existing held-out check is still there


def test_train_recipe_output_unchanged_without_eval_batches():
    out = _run_world(["--model", "resnet20", "--steps", "2", "--batch", "16"], "recipes/PyTorch-GPU/train_resnet50.py")
    assert "eval" not in out


def test_score_recipe_tiny_world2_writes_both_rank_files(tmp_path):
    out = _run_world(["--model", "tiny", "--synthetic", "64", "--image", "32", "--batch", "16", "--out", str(tmp_path)],
                     "recipes/PyTorch-GPU/score_resnet50.py")
    import numpy as np
    parts = [np.load(tmp_path / f"top5.rank{r}.npy") for r in range(2)]
    assert [p.shape for p in parts] == [(32, 5), (32, 5)]
    assert all(((p >= 0) & (p < 10)).all() for p in parts)
    assert out["images"] == 64 and out["world"] == 2 and out["transport"] == "stub" and 0 <= out["top1"] <= out["top5"] <= 1, out


def test_score_job_variant_dry_runs(tmp_path, monkeypatch):
    from click.testing import CliRunner
    from batch_shipyard_b200 import cli
    monkeypatch.setenv("SHIPYARD_STATE_DIR", str(tmp_path / "state"))
    res = CliRunner().invoke(cli.cli, ["jobs", "add", "--configdir", os.path.join(ROOT, "recipes", "PyTorch-GPU", "config", "score"),
                                       "--dry-run", "--raw"], obj=cli.CliContext())
    assert res.exit_code == 0, res.output
    dry = json.loads(res.output)["score"]
    assert dry["dry_run"] and "score_resnet50.py" in json.dumps(dry)
