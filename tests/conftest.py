import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with `-m gpu` under gpurun)")
    config.addinivalue_line("markers", "multigpu: needs >= 2 GPUs")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        ngpu = torch.cuda.device_count() if torch.cuda.is_available() else 0
    except Exception:
        ngpu = 0
    for item in items:
        if "gpu" in item.keywords and ngpu == 0:
            item.add_marker(pytest.mark.skip(reason="no GPU on this box"))
        if "multigpu" in item.keywords and ngpu < 2:
            item.add_marker(pytest.mark.skip(reason="needs >= 2 GPUs"))


@pytest.fixture(autouse=True)
def _cpu_tests_see_no_gpu(request, monkeypatch):
    """A test not marked `gpu` models a CPU-only box, where pools get virtual CPU-slot nodes (`cpu-<i>`).  On a machine with GPUs
    the local backend would make one node per GPU and refuse a pool with more nodes than GPUs, so these tests see zero GPUs
    whatever the machine has (the GPU probe honours SHIPYARD_FAKE_GPUS; a test may set its own count)."""
    if "gpu" in request.keywords:
        yield
        return
    from batch_shipyard_b200.pool import topology
    monkeypatch.setenv("SHIPYARD_FAKE_GPUS", "0")
    topology.probe(refresh=True)
    yield
    topology._CACHE = None                     # the next probe reads the real machine again


@pytest.fixture(scope="session", autouse=True)
def _native_executables():
    """Built artefacts are not in the history (see .gitignore); the libraries build themselves on first load (ops/*.py), the
    executables a recipe command names by path (`shipyard-mpibench`, `shipyard-diskbench`) are built here.  A no-op when they
    are already up to date, which is the case after `python native/build.py` / `__graft_entry__.build()`."""
    from batch_shipyard_b200._build import ensure_built, native_dir
    want = {"taskrun": "shipyard-taskrun", "gpuprobe": "shipyard-gpuprobe", "mpibench": "shipyard-mpibench", "diskbench": "shipyard-diskbench"}
    missing = [k for k, exe in want.items() if not os.path.exists(os.path.join(native_dir(), exe))]
    if "mpibench" in missing:
        missing = ["coll", "mpi"] + missing                          # link-time dependencies (native/build.py DEPS)
    if missing:
        ensure_built(missing)
