"""The full-document YAML examples in the reference's configuration guides (docs/11..18) validate against our schemas.

The examples are stored under tests/golden/reference (guide_yaml_examples.json, taken from Batch Shipyard 3.9.1).
Two examples contain typos that the reference's own schema rejects as well (`polling_interval.jobs` in the federation guide,
`preempty_type` in the Slurm guide); those keys are removed before validation."""
import json
import os

import pytest
import yaml

from batch_shipyard_b200.config.schema import ConfigType, validate

with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference", "guide_yaml_examples.json")) as _f:
    EXAMPLES = json.load(_f)
CASES = [("11-batch-shipyard-configuration-credentials.md", ConfigType.Credentials, ("credentials",)),
         ("13-batch-shipyard-configuration-pool.md", ConfigType.Pool, ("pool_specification",)),
         ("14-batch-shipyard-configuration-jobs.md", ConfigType.Jobs, ("job_specifications",)),
         ("15-batch-shipyard-configuration-fs.md", ConfigType.RemoteFS, ("remote_fs",)),
         ("16-batch-shipyard-configuration-monitor.md", ConfigType.Monitor, ("monitoring",)),
         ("17-batch-shipyard-configuration-federation.md", ConfigType.Federation, ("federation",)),
         ("18-batch-shipyard-configuration-slurm.md", ConfigType.Slurm, ("slurm",))]


def _strip_doc_typos(ct, data):
    if ct is ConfigType.Federation:
        (((data.get("federation") or {}).get("proxy_options") or {}).get("polling_interval") or {}).pop("jobs", None)
    if ct is ConfigType.Slurm:
        for part in ((((data.get("slurm") or {}).get("slurm_options") or {}).get("elastic_partitions")) or {}).values():
            part.pop("preempty_type", None)


@pytest.mark.parametrize("doc,ct,roots", CASES, ids=[c[0][:2] for c in CASES])
def test_reference_guide_examples_validate(doc, ct, roots):
    n = 0
    for b in EXAMPLES[doc]:
        try:
            data = yaml.safe_load(b)
        except yaml.YAMLError:
            continue
        if not isinstance(data, dict) or not any(r in data for r in roots):
            continue
        _strip_doc_typos(ct, data)
        validate(ct, data, source=doc)             # raises ValidationError listing every problem
        n += 1
    assert n >= 1
