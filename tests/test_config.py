"""Config layer: schema DSL, validation strictness, discovery, merge order, settings defaults."""
import json
import os

import pytest
import yaml

from batch_shipyard_b200.config import loader, settings as S
from batch_shipyard_b200.config.schema import ConfigType, ValidationError, compile_schema, validate
from batch_shipyard_b200.utils import util

REF_TEMPLATES = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference", "config_templates")   # Batch Shipyard 3.9.1


@pytest.mark.parametrize("ct,name", [(ConfigType.Credentials, "credentials"), (ConfigType.Global, "config"), (ConfigType.Pool, "pool"),
                                     (ConfigType.Jobs, "jobs"), (ConfigType.RemoteFS, "fs"), (ConfigType.Monitor, "monitor"),
                                     (ConfigType.Federation, "federation"), (ConfigType.Slurm, "slurm")])
def test_reference_templates_validate(ct, name):
    with open(os.path.join(REF_TEMPLATES, name + ".yaml")) as f:
        validate(ct, yaml.safe_load(f))


def test_schema_strictness():
    with pytest.raises(ValidationError) as e:
        validate(ConfigType.Pool, {"pool_specification": {"id": "p", "vm_sizee": "x"}})
    assert "unknown key" in str(e.value)
    with pytest.raises(ValidationError) as e:
        validate(ConfigType.Pool, {"pool_specification": {"vm_size": "x"}})
    assert "required key missing" in str(e.value)
    with pytest.raises(ValidationError):
        validate(ConfigType.Pool, {"pool_specification": {"id": "p", "node_fill_type": "stack"}})
    with pytest.raises(ValidationError):
        validate(ConfigType.Pool, {"pool_specification": {"id": "p", "max_tasks_per_node": 0}})
    with pytest.raises(ValidationError):
        validate(ConfigType.Jobs, {"job_specifications": [{"id": "j", "tasks": [{"multi_instance": {"num_instances": 2, "mpi": {"runtime": "lam", "processes_per_node": 1}}}]}]})
    # null is "absent" everywhere optional
    validate(ConfigType.Pool, {"pool_specification": {"id": "p", "autoscale": None, "ssh": None}})


def test_schema_dsl():
    n = compile_schema({"a!": "int:0..3", "b": ["str"], "c": {"*": "bool"}, "d": "int|str", "e": "enum:x|y"})
    from batch_shipyard_b200.config.schema import _check
    errs = []
    _check(n, {"a": 5, "b": [1, "x"], "c": {"k": "no"}, "d": [1], "e": "z"}, "$", errs)
    assert len(errs) == 4 and any("maximum" in x for x in errs)


def test_merge_and_discovery(tmp_path, monkeypatch):
    d = tmp_path / "conf"
    d.mkdir()
    (d / "config.yaml").write_text("batch_shipyard:\n  storage_entity_prefix: abc\nglobal_resources:\n  docker_images: [a, b]\n")
    (d / "pool.json").write_text(json.dumps({"pool_specification": {"id": "p1", "vm_count": {"dedicated": 2}}}))
    other = tmp_path / "jobs-explicit.yaml"
    other.write_text("job_specifications:\n- id: j1\n  tasks:\n  - docker_image: a\n    command: echo\n")
    monkeypatch.setenv("SHIPYARD_JOBS_CONF", str(other))
    cfg = loader.load_configs(configdir=str(d))
    assert cfg["pool_specification"]["id"] == "p1" and cfg["job_specifications"][0]["id"] == "j1"
    assert cfg["_config_files"]["pool"].endswith("pool.json")
    with pytest.raises(loader.ConfigError):
        loader.load_configs(configdir=str(d), required=(ConfigType.Federation,))
    (d / "fs.yaml").write_text("remote_fs:\n  bogus: 1\n")
    with pytest.raises(loader.ConfigError) as e:
        loader.load_configs(configdir=str(d))
    assert "unknown key" in str(e.value)


def test_merge_dict_lists_replace():
    a = {"x": {"y": [1, 2], "z": 1}, "k": 1}
    b = {"x": {"y": [3]}, "n": 2}
    assert util.merge_dict(a, b) == {"x": {"y": [3], "z": 1}, "k": 1, "n": 2}


def test_show_config_masks_secrets():
    out = loader.dump_config({"credentials": {"storage": {"s": {"account_key": "SECRET", "account": "acc"}}}, "_raw": True})
    assert "SECRET" not in out and "acc" in out and "_raw" not in out


def test_pool_settings_defaults_and_rules():
    ps = S.pool_settings({"pool_specification": {"id": "p"}})
    assert ps.max_tasks_per_node == 1 and ps.block_until_all_global_resources_loaded and not ps.inter_node_communication_enabled
    assert ps.ssh_expiry_days == 30 and ps.rac_starting_port == 49000 and ps.container_runtimes_default == "runc"
    assert ps.node_fill_type == "pack" and ps.upload_diagnostics_logs_on_unusable
    with pytest.raises(ValueError):
        S.pool_settings({"pool_specification": {"id": "p", "remote_access_control": {"starting_port": 50000}}})
    with pytest.raises(ValueError):
        S.pool_settings({"pool_specification": {"id": "p", "autoscale": {"evaluation_interval": "00:01:00", "formula": "x"}}})


def test_gpu_size_classification():
    assert S.is_gpu_pool("B200x8") and S.local_gpu_count_from_vm_size("b200x4") == 4 and S.is_rdma_pool("B200x8")
    assert S.is_gpu_pool("STANDARD_NC6") and S.is_gpu_pool("STANDARD_ND96isr_H100_v5") and not S.is_gpu_pool("STANDARD_D2_V2")
    assert S.is_rdma_pool("STANDARD_HC44rs") and not S.is_rdma_pool("STANDARD_D2_V2")


def test_num_instances_keywords():
    assert S.resolve_num_instances("pool_current_dedicated", 3, 1, 5, 2) == 3
    assert S.resolve_num_instances("pool_specification_vm_count_low_priority", 3, 1, 5, 2) == 2   # (the reference crashes here: Q2)
    assert S.resolve_num_instances(4, 0, 0, 0, 0) == 4
    with pytest.raises(ValueError):
        S.resolve_num_instances("everything", 1, 1, 1, 1)


def test_timedelta_and_helpers():
    assert util.convert_string_to_timedelta("1.12:30:05").total_seconds() == 86400 + 12 * 3600 + 30 * 60 + 5
    assert util.timedelta_to_string(util.convert_string_to_timedelta("02:00:00")) == "02:00:00"
    with pytest.raises(ValueError):
        util.convert_string_to_timedelta("2 hours")
    assert util.wrap_commands_in_shell(["a", "b"]).startswith("/bin/bash -c 'set -e; set -o pipefail; a; b; wait'")
    assert util.singularity_image_name_on_disk("docker://busybox") == "busybox_latest.sif"
    assert util.singularity_image_name_on_disk("shub://singularityhub/busybox") == "singularityhub-busybox_master.sif"
    assert util.parse_size_to_mb("2g") == 2048 and util.parse_size_to_mb("512m") == 512
    assert util.ip_from_address_prefix("10.0.0.0/29") == ["10.0.0.4", "10.0.0.5", "10.0.0.6"]
