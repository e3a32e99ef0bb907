"""GPU collectives: every kernel vs a PyTorch fp64 reference, 1 GPU and (when present) 2/4/8 GPUs."""
import pytest
import torch

from _mp import run_ranks

pytestmark = pytest.mark.gpu


def _ngpu():
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


def _need_multi():
    if _ngpu() < 2:
        pytest.skip("needs at least 2 GPUs on the box")


def test_single_gpu_collectives():
    ok, outs = run_ranks("_coll_worker.py", 1, extra=["--quick"], gpu=True, timeout=300)
    assert ok, "\n".join(o[-3000:] for o in outs)
    assert "transport=p2p" in outs[0] or "transport=nvls" in outs[0]


@pytest.mark.multigpu
@pytest.mark.parametrize("transport", ["auto", "p2p"])
def test_multi_gpu_collectives(transport):
    _need_multi()
    world = min(_ngpu(), 8)
    import os
    extra = ["--transport", transport] + (["--quick"] if os.environ.get("SHIPYARD_TEST_QUICK") else [])
    ok, outs = run_ranks("_coll_worker.py", world, extra=extra, gpu=True, timeout=600)
    assert ok, "\n".join(o[-3000:] for o in outs)


@pytest.mark.multigpu
def test_nccl_preload_shim_under_torch_distributed(tmp_path):
    """LD_PRELOAD the shim under a torchrun NCCL job: results stay correct and the collectives ran on our kernels."""
    _need_multi()
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    shim = os.path.join(root, "batch_shipyard_b200", "_native", "libshipyard_preload.so")
    assert os.path.exists(shim), "libshipyard_preload.so is not built"
    world = min(_ngpu(), 8)
    env = dict(os.environ, LD_PRELOAD=shim, SHIPYARD_PRELOAD_STATS="1", SHIPYARD_COLL_SESSION="preloadtest")
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
                        "--master-port", "29577", os.path.join(root, "tests", "_preload_worker.py")], env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True, timeout=600)
    (tmp_path / "preload_test.log").write_text(p.stdout)
    assert p.returncode == 0, p.stdout[-6000:]
    assert p.stdout.count("ok=True") == world


@pytest.mark.multigpu
@pytest.mark.parametrize("transport", ["auto", "p2p"])
def test_k10_gemm_allreduce_fused(transport):
    _need_multi()
    world = min(_ngpu(), 8)
    ok, outs = run_ranks("_k10_worker.py", world, extra=["--transport", transport], gpu=True, timeout=600)
    assert ok, "\n".join(o[-3000:] for o in outs)


@pytest.mark.multigpu
def test_flag_protocol_litmus_over_nvlink():
    """Message-passing litmus on P2P-mapped flags (payload stores, release flag / acquire flag, payload loads), 500 ping-pong rounds."""
    _need_multi()
    ok, outs = run_ranks("_litmus_worker.py", 2, extra=["--rounds", "500"], gpu=True, timeout=300)
    assert ok, "\n".join(o[-3000:] for o in outs)
    assert all("transport=gpu" in o for o in outs)


@pytest.mark.multigpu
def test_data_parallel_trainer_equals_single_gpu(tmp_path):
    """N ranks x the same batch: the averaged gradient equals the 1-GPU gradient, so the parameters after 3 steps of the fused
    all-reduce + SGD kernel must equal the 1-GPU run (full ResNet-50, CUDA graph, NVLS / P2P transport).  Different per-rank data is
    not comparable with a single large batch (BatchNorm statistics are per rank); the collectives' numerics with different data per
    rank are covered by test_multi_gpu_collectives."""
    _need_multi()
    world = min(_ngpu(), 8)
    ref = str(tmp_path / "ref.pt")
    ok, outs = run_ranks("_trainer_worker.py", 1, extra=["--ref", ref], gpu=True, timeout=600)
    assert ok, outs[0][-3000:]
    ok, outs = run_ranks("_trainer_worker.py", world, extra=["--ref", ref], gpu=True, timeout=900,
                         env={"SHIPYARD_COLL_TIMEOUT_MS": "180000"})
    assert ok, "\n".join(o[-3000:] for o in outs)
