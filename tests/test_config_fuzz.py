"""Mutation fuzzing of valid configurations: a config either fails validation with a ValidationError, or every settings accessor and
the job builder's dry run either work or raise a ValueError / KeyError / RuntimeError with a message (which the CLI prints as
`ERROR: ...`) — never an AttributeError / TypeError from deep inside.  Deterministic seeds, a few hundred mutations."""
import copy
import os
import random

def _read(path):
    with open(path) as f:
        return f.read()


import pytest
import yaml

from batch_shipyard_b200.backend.local import LocalBackend
from batch_shipyard_b200.config import loader, settings as S
from batch_shipyard_b200.config.schema import ConfigType, ValidationError, validate
from batch_shipyard_b200.jobs import submit
from batch_shipyard_b200.pool import autoscale, provision
from batch_shipyard_b200.utils.util import merge_dict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VALUES = [None, 0, -1, "", "x", True, [], {}, [1], {"a": 1}, 3.5, "00:00:01", "pool_current_dedicated", "1", 10 ** 9, "auto", [None]]
BATCH = (ConfigType.Credentials, ConfigType.Global, ConfigType.Pool, ConfigType.Jobs)


def _paths(node, pre=()):
    out = []
    if isinstance(node, dict):
        for k, v in node.items():
            out.append(pre + (k,)); out += _paths(v, pre + (k,))
    elif isinstance(node, list):
        for i, v in enumerate(node):
            out.append(pre + (i,)); out += _paths(v, pre + (i,))
    return out


def _mutate(rng, cfg):
    p = rng.choice(_paths(cfg))
    node = cfg
    for k in p[:-1]:
        node = node[k]
    if rng.random() < 0.3:
        node.pop(p[-1])
    else:
        node[p[-1]] = copy.deepcopy(rng.choice(VALUES))
    return p


@pytest.mark.parametrize("recipe", ["PyTorch-GPU", "mpiBench-OpenMPI", "HPCG-Infiniband-IntelMPI", "TensorFlow-Distributed"])
def test_mutated_recipe_configs_fail_cleanly(recipe, tmp_path):
    rng = random.Random(sum(map(ord, recipe)))
    d = os.path.join(ROOT, "recipes", recipe, "config")
    datas = {k: yaml.safe_load(_read(os.path.join(d, k.value + ".yaml"))) for k in BATCH if os.path.exists(os.path.join(d, k.value + ".yaml"))}
    crashes = []
    for it in range(120):
        ds = copy.deepcopy(datas)
        kind = rng.choice(list(ds))
        path = _mutate(rng, ds[kind])
        try:
            for k, v in ds.items():
                validate(k, loader.normalize(k, v))
        except ValidationError:
            continue
        except Exception as e:  # noqa: BLE001
            crashes.append(("validate", kind.value, path, repr(e)[:120])); continue
        cfg = {}
        for k in BATCH:
            if k in ds:
                cfg = merge_dict(cfg, ds[k])
        try:
            S.pool_settings(cfg); S.global_settings(cfg)
            provision.adjust_settings_for_pool_creation(cfg)
            submit.add_jobs(LocalBackend(state_dir=str(tmp_path / f"s{it}")), cfg, dry_run=True)
        except (ValueError, KeyError, RuntimeError):
            continue
        except Exception as e:  # noqa: BLE001
            crashes.append(("settings/builder", kind.value, path, repr(e)[:120]))
    assert crashes == [], crashes


def test_mutated_reference_templates_fail_cleanly():
    rng = random.Random(7)
    kinds = {ConfigType.Pool: "pool", ConfigType.Global: "config", ConfigType.Credentials: "credentials", ConfigType.RemoteFS: "fs",
             ConfigType.Slurm: "slurm", ConfigType.Federation: "federation", ConfigType.Monitor: "monitor"}
    templates = os.path.join(ROOT, "tests", "golden", "reference", "config_templates")          # Batch Shipyard 3.9.1
    datas = {k: yaml.safe_load(_read(os.path.join(templates, v + ".yaml"))) for k, v in kinds.items()}
    crashes = []
    for _ in range(500):
        ds = copy.deepcopy(datas)
        kind = rng.choice(list(ds))
        path = _mutate(rng, ds[kind])
        try:
            for k, v in ds.items():
                validate(k, loader.normalize(k, v))
        except ValidationError:
            continue
        except Exception as e:  # noqa: BLE001
            crashes.append(("validate", kind.value, path, repr(e)[:120])); continue
        cfg = {}
        for v in ds.values():
            cfg = merge_dict(cfg, v)
        for name, fn in (("pool", lambda: (S.pool_settings(cfg), provision.adjust_settings_for_pool_creation(cfg))),
                         ("autoscale", lambda: autoscale.generate_formula(S.pool_settings(cfg))
                          if S.pool_settings(cfg).autoscale and S.pool_settings(cfg).autoscale.scenario else None),
                         ("global", lambda: S.global_settings(cfg)), ("fs", lambda: S.remotefs_storage_clusters(cfg)),
                         ("slurm", lambda: S.slurm_options(cfg))):
            try:
                fn()
            except (ValueError, KeyError, RuntimeError):
                pass
            except Exception as e:  # noqa: BLE001
                crashes.append((name, kind.value, path, repr(e)[:120]))
    assert crashes == [], crashes
