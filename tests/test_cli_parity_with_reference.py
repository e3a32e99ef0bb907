"""Option-by-option comparison of the click command tree with the reference's `shipyard.py`.

The reference's commands, their options, its SHIPYARD_* environment variables and the `--raw` capable commands of its usage guide
are stored in tests/golden/reference/cli.json (Batch Shipyard 3.9.1, see make_golden.py there)."""
import json
import os

import click

from batch_shipyard_b200 import cli

with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference", "cli.json")) as _f:
    REF = json.load(_f)
# options every command gets through shared decorators on both sides
COMMON = {"--configdir", "--credentials", "--config", "--pool", "--jobs", "--fs", "--monitor", "--federation", "--slurm", "--raw", "--yes",
          "--verbose", "--show-config"}


def _ours():
    out = {}

    def walk(g, path):
        for n, c in g.commands.items():
            if isinstance(c, click.Group):
                walk(c, path + [n])
            else:
                out[tuple(path + [n])] = {o for p in c.params if isinstance(p, click.Option) for o in p.opts if o.startswith("--")}
    walk(cli.cli, [])
    return out


def test_every_reference_option_exists_on_the_same_command():
    blocks = REF["commands"]
    assert len(blocks) == 105
    ours = _ours()
    assert len(ours) == 105
    missing = []
    for grp, name, fn, ref_opts in blocks:
        opts = set(ref_opts) - COMMON
        # the function name spells the command path: fed_jobs_del -> ("fed", "jobs", "del"); names keep their dashes
        # (sub-group commands drop the top group: nodes_count is `pool nodes count`, sas_create is `storage sas create`)
        joined = {k: "_".join(k).replace("-", "_") for k in ours}
        cands = ([k for k, j in joined.items() if j == fn] or [k for k, j in joined.items() if j.endswith("_" + fn) and k[-2] == grp]
                 or [k for k in ours if k[-1] == name and k[-2] == grp])                     # e.g. misc_mirror is `misc mirror-images`
        assert len(cands) == 1, (fn, cands)
        lost = sorted(o for o in opts if o not in ours[cands[0]])
        if lost:
            missing.append((" ".join(cands[0]), lost))
    assert missing == [], missing


def test_raw_capable_commands_and_environment_variables_of_the_usage_guide_exist():
    """docs/20-batch-shipyard-usage.md lists the ~30 commands that support --raw and the SHIPYARD_* variables of the CLI."""
    listed = [tuple(m.split()) for m in REF["raw_commands"]]
    assert len(listed) >= 30
    ours = _ours()
    assert [c for c in listed if c not in ours] == []
    src = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "batch_shipyard_b200", "cli.py")).read()
    env = set(REF["envvars"])
    assert len(env) >= 20 and sorted(e for e in env if e not in src) == []
