"""Every key path of the reference's pykwalify schemas is accepted by our schemas.

Only key NAMES and nesting are compared (our notation for types / enums is different on purpose).  The reference's key paths and
enumerations are stored in tests/golden/reference/schemas.json (Batch Shipyard 3.9.1, see make_golden.py there)."""
import json
import os

def _read(path):
    with open(path) as f:
        return f.read()


import pytest
import yaml

with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference", "schemas.json")) as _f:
    REF = json.load(_f)
OURS = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "batch_shipyard_b200", "config", "schemas")


def _our_paths(node, prefix=""):
    out = set()
    if isinstance(node, dict):
        for k, v in node.items():
            p = f"{prefix}.{str(k).rstrip('!')}" if prefix else str(k).rstrip("!")
            out.add(p)
            out |= _our_paths(v, p)
    elif isinstance(node, list):
        for v in node:
            out |= _our_paths(v, prefix + "[]")
    return out


@pytest.mark.parametrize("name", ["credentials", "config", "pool", "jobs", "fs", "monitor", "federation", "slurm"])
def test_reference_schema_keys_are_accepted(name):
    ref = set(REF[name]["key_paths"])
    ours = _our_paths(yaml.safe_load(_read(os.path.join(OURS, name + ".yaml"))))

    def covered(p):                                   # a named key of the reference may be served by a "*" (any key) entry of ours
        parts = p.split(".")
        return p in ours or any(".".join(parts[:i] + ["*"] + parts[i + 1:]) in ours for i in range(len(parts)))

    missing = sorted(p for p in ref if not covered(p))
    assert missing == [], missing
    assert len(ref) > 40


def _our_specs(node, prefix="", out=None):
    out = {} if out is None else out
    if isinstance(node, dict):
        for k, v in node.items():
            p = f"{prefix}.{str(k).rstrip('!')}" if prefix else str(k).rstrip("!")
            if isinstance(v, str):
                out[p] = v
            else:
                _our_specs(v, p, out)
    elif isinstance(node, list):
        for v in node:
            if isinstance(v, str):
                out[prefix + "[]"] = v
            else:
                _our_specs(v, prefix + "[]", out)
    return out


@pytest.mark.parametrize("name", ["credentials", "config", "pool", "jobs", "fs", "monitor", "federation", "slurm"])
def test_reference_enums_are_enums_here_with_at_least_the_same_values(name):
    """Where the reference restricts a key to an enumeration, so do we (strictness parity), and every reference value is accepted."""
    import re
    ref = {path: set(values) for path, values in REF[name]["enums"].items()}
    ours = _our_specs(yaml.safe_load(_read(os.path.join(OURS, name + ".yaml"))))
    problems = []
    for path, values in ref.items():
        parts = path.split(".")
        spec = ours.get(path) or next((ours[q] for i in range(len(parts)) if (q := ".".join(parts[:i] + ["*"] + parts[i + 1:])) in ours), None)
        m = re.search(r"enum:([^\s\]]+)", spec or "")
        if not m:
            problems.append((path, "not an enum here", spec))
        elif not values <= set(m.group(1).split("|")):
            problems.append((path, "missing values", sorted(values - set(m.group(1).split("|")))))
    assert problems == [], problems
