"""Every configuration file of every reference recipe (`recipes/*/config/*.yaml`, 134 files) passes our loader's
normalisation + strict validation unchanged — what a user gets when pointing `--configdir` at a recipe they already have.
The recipes' config directories of Batch Shipyard 3.9.1 are stored unchanged under tests/golden/reference/recipes."""
import os

def _read(path):
    with open(path) as f:
        return f.read()


import yaml

from batch_shipyard_b200.config import loader
from batch_shipyard_b200.config.schema import ConfigType, validate

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference", "recipes")
KINDS = {"credentials": ConfigType.Credentials, "config": ConfigType.Global, "pool": ConfigType.Pool, "jobs": ConfigType.Jobs,
         "fs": ConfigType.RemoteFS, "monitor": ConfigType.Monitor, "federation": ConfigType.Federation, "slurm": ConfigType.Slurm}


def _files():
    out = []
    for d, _, fs in os.walk(ROOT):
        for f in sorted(fs):
            base, ext = os.path.splitext(f)
            if ext in (".yaml", ".yml") and base in KINDS and os.path.basename(d) == "config":
                out.append(os.path.join(d, f))
    return sorted(out)


def test_all_reference_recipe_configs_validate():
    files = _files()
    assert len(files) >= 130
    problems = []
    for p in files:
        kind = KINDS[os.path.splitext(os.path.basename(p))[0]]
        try:
            validate(kind, loader.normalize(kind, yaml.safe_load(_read(p))), source=p)
        except Exception as e:  # noqa: BLE001
            problems.append((os.path.relpath(p, ROOT), str(e)[:300]))
    assert problems == [], problems


def test_optional_processes_per_node_and_legacy_auto_scratch():
    """The two spellings the OpenFOAM recipes of the reference rely on."""
    from batch_shipyard_b200.config import settings as S
    from batch_shipyard_b200.jobs import mpi as M
    m = M.mpi_settings({"runtime": "openmpi"})
    assert m.processes_per_node is None
    line, _ = M.construct_mpi_command(m, 4, "app")
    assert "-np" not in line and "ppr:" not in line and line.endswith(" app")
    assert M.resolve_processes_per_node(None, 8) == 1
    jobs = loader.normalize(ConfigType.Jobs, {"job_specifications": [{"id": "j", "auto_scratch": True, "tasks": [{"command": "x"}]}]})
    a = S.job_auto_scratch(jobs["job_specifications"][0])
    assert a is not None and a.setup == "dependency"
    off = loader.normalize(ConfigType.Jobs, {"job_specifications": [{"id": "j", "auto_scratch": False, "tasks": []}]})
    assert "auto_scratch" not in off["job_specifications"][0]


def test_every_reference_recipe_dry_runs_through_the_job_builder(tmp_path, monkeypatch):
    """`shipyard jobs add --dry-run` on the reference's own recipe directories (their pool / jobs / config files, untouched): task-factory
    expansion, image policy, container option synthesis, MPI launcher line, multi-instance settings and data-movement specs all resolve."""
    from batch_shipyard_b200.backend.local import LocalBackend
    from batch_shipyard_b200.jobs import submit
    monkeypatch.setenv("SHIPYARD_STATE_DIR", str(tmp_path / "state"))
    skip = (ConfigType.RemoteFS, ConfigType.Monitor, ConfigType.Federation, ConfigType.Slurm)
    done, problems = 0, []
    for recipe in sorted(os.listdir(ROOT)):
        cfgd = os.path.join(ROOT, recipe, "config")
        if not os.path.isdir(cfgd):
            continue
        variants = [cfgd] if os.path.exists(os.path.join(cfgd, "jobs.yaml")) else \
            [os.path.join(cfgd, v) for v in sorted(os.listdir(cfgd)) if os.path.isdir(os.path.join(cfgd, v))]
        for v in variants:
            if not os.path.exists(os.path.join(v, "jobs.yaml")):
                continue
            try:
                cfg = loader.load_configs({}, v, skip=skip)
                cfg.setdefault("credentials", {"storage": {"mystorageaccount": {"account": "local"}}})
                out = submit.add_jobs(LocalBackend(state_dir=str(tmp_path / f"s{done}")), cfg, dry_run=True)
                assert out and all(j.get("dry_run") for j in out.values())
                done += 1
            except Exception as e:  # noqa: BLE001
                problems.append((os.path.relpath(v, ROOT), f"{type(e).__name__}: {e}"[:300]))
    assert problems == [], problems
    assert done >= 50
