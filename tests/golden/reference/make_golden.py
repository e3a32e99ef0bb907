#!/usr/bin/env python3
"""Regenerate the Batch Shipyard 3.9.1 fixtures in this directory from a checkout of Azure/batch-shipyard.

    python tests/golden/reference/make_golden.py /path/to/batch-shipyard

Configuration files (recipe configs, config templates) are copied unchanged.  From the schemas, the CLI module and the
usage / configuration guides only what the parity tests compare against is kept: schema key paths and enumerations,
command options and environment variables, the YAML examples and the list of `--raw` capable commands."""
import json
import os
import re
import shutil
import sys

import yaml

HERE = os.path.dirname(os.path.abspath(__file__))
SCHEMAS = ["credentials", "config", "pool", "jobs", "fs", "monitor", "federation", "slurm"]
GUIDES = ["11-batch-shipyard-configuration-credentials.md", "13-batch-shipyard-configuration-pool.md",
          "14-batch-shipyard-configuration-jobs.md", "15-batch-shipyard-configuration-fs.md",
          "16-batch-shipyard-configuration-monitor.md", "17-batch-shipyard-configuration-federation.md",
          "18-batch-shipyard-configuration-slurm.md"]


def _read(path):
    with open(path) as f:
        return f.read()


def _key(k):
    return "*" if str(k).startswith(("regex;", "re;")) else str(k)


def schema_paths(node, prefix=""):
    """Every key path of a pykwalify schema (`a.b[].c`; regex keys become `*`)."""
    out = set()
    if not isinstance(node, dict):
        return out
    if "mapping" in node or node.get("type") == "map":
        for k, v in (node.get("mapping") or {}).items():
            p = f"{prefix}.{_key(k)}" if prefix else _key(k)
            out.add(p)
            out |= schema_paths(v, p)
    if "sequence" in node or node.get("type") == "seq":
        for v in node.get("sequence") or []:
            out |= schema_paths(v, prefix + "[]")
    return out


def schema_enums(node, prefix="", out=None):
    """{key path: enumeration values} of a pykwalify schema."""
    out = {} if out is None else out
    if not isinstance(node, dict):
        return out
    if "enum" in node:
        out[prefix] = sorted({str(v) for v in node["enum"]})
    if "mapping" in node or node.get("type") == "map":
        for k, v in (node.get("mapping") or {}).items():
            schema_enums(v, f"{prefix}.{_key(k)}" if prefix else _key(k), out)
    if "sequence" in node or node.get("type") == "seq":
        for v in node.get("sequence") or []:
            schema_enums(v, prefix + "[]", out)
    return out


def _dump(name, data):
    with open(os.path.join(HERE, name), "w") as f:
        json.dump(data, f, indent=1, sort_keys=True)
        f.write("\n")


def main(ref):
    for sub in ("config_templates", "recipes"):
        shutil.rmtree(os.path.join(HERE, sub), ignore_errors=True)
    shutil.copytree(os.path.join(ref, "config_templates"), os.path.join(HERE, "config_templates"))
    for recipe in sorted(os.listdir(os.path.join(ref, "recipes"))):
        src = os.path.join(ref, "recipes", recipe, "config")
        if os.path.isdir(src):
            shutil.copytree(src, os.path.join(HERE, "recipes", recipe, "config"))

    schemas = {}
    for name in SCHEMAS:
        node = yaml.safe_load(_read(os.path.join(ref, "schemas", name + ".yaml")))
        schemas[name] = {"key_paths": sorted(schema_paths(node)), "enums": schema_enums(node)}
    _dump("schemas.json", schemas)

    _dump("guide_yaml_examples.json",
          {doc: re.findall(r"```yaml\n(.*?)```", _read(os.path.join(ref, "docs", doc)), flags=re.S) for doc in GUIDES})

    src = _read(os.path.join(ref, "shipyard.py"))
    commands = [[grp, name, fn, sorted(set(re.findall(r"@click\.option\(\s*'(--[\w-]+)'", decos)))]
                for grp, name, decos, fn in re.findall(r"@(\w+)\.command\('([\w-]+)'\)(.*?)\ndef (\w+)\(", src, flags=re.S)]
    usage = _read(os.path.join(ref, "docs", "20-batch-shipyard-usage.md"))
    block = usage[usage.index("The following commands support this option:"):usage.index("`--show-config` will output")]
    _dump("cli.json", {"commands": commands,
                       "raw_commands": re.findall(r"\* `([a-z \-]+)`", block),
                       "envvars": sorted(set(re.findall(r"envvar='(SHIPYARD_[A-Z_]+)'", src)))})


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
