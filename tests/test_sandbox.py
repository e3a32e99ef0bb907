"""Process sandbox of shipyard-taskrun: the container semantics of the reference's run-option synthesis
(/root/reference/convoy/settings.py:3875-3901, 3919-4051, 4374-4443) enforced without a container runtime."""
import json
import os
import subprocess
import time

import pytest

from _helpers import make, read, run, up
from batch_shipyard_b200.backend import runspec


def _sandbox_mode():
    """What this box allows: mountns (root), userns (unprivileged user namespaces) or none."""
    if os.geteuid() == 0:
        return "mountns" if subprocess.call(["unshare", "-m", "true"], stderr=subprocess.DEVNULL) == 0 else "none"
    return "userns" if subprocess.call(["unshare", "-Urm", "true"], stderr=subprocess.DEVNULL) == 0 else "none"


MODE = _sandbox_mode()
needs_ns = pytest.mark.skipif(MODE == "none", reason="box allows neither mount nor user namespaces")


def _result(b, job, task):
    with open(b.task_file_path(job, task, "result.json")) as f:
        return json.load(f)


@needs_ns
def test_data_volume_bind_and_private_tmp(tmp_path, monkeypatch):
    monkeypatch.setenv("SHIPYARD_SANDBOX_PRIVATE_TMP", "1")          # a container's own /tmp (opt-in; TMPDIR is always private)
    host = tmp_path / "hostdata"
    host.mkdir()
    (host / "in.txt").write_text("payload")
    # the bind exists only inside the task's mount namespace.  A mount point is created on the real file system first, so without
    # root (user namespace) the container path must lie where the user may create a directory: the file-system root needs root.
    mnt = f"/shipyard-test-mnt-{os.getpid()}" if os.geteuid() == 0 else str(tmp_path / "container" / "shipyard-test-mnt")
    extra = {"global_resources": {"volumes": {"data_volumes": {
        "dv": {"host_path": str(host), "container_path": mnt},
        "ro": {"host_path": str(host), "container_path": mnt + "-ro", "bind_options": "ro"},
        "anon": {"container_path": mnt + "-anon"}}}}}
    tasks = [{"id": "t", "docker_image": "busybox", "data_volumes": ["dv", "ro", "anon"],
              "command": f"cat {mnt}/in.txt; echo out > {mnt}/out.txt; touch {mnt}-ro/x 2>/dev/null && echo RO-WRITABLE; "
                         f"echo scratch > {mnt}-anon/a; echo tmp > /tmp/only-in-container; echo mode=$SHIPYARD_SANDBOX"}]
    cfg, b = make(tmp_path, tasks=tasks, extra=extra)
    up(cfg, b)
    run(cfg, b)
    out = read(b, "job1", "t")
    assert "payload" in out and "RO-WRITABLE" not in out and f"mode={MODE}" in out
    assert (host / "out.txt").read_text().strip() == "out"          # rw bind reaches the host directory
    assert not os.path.exists(mnt) or not os.listdir(mnt)                        # the mount point is not populated outside
    assert not os.path.exists("/tmp/only-in-container")               # private /tmp
    assert _result(b, "job1", "t")["sandbox"] == MODE
    # --rm (remove_container_after_exit defaults to true): the container scratch (private tmp, anonymous volume) is gone
    tdir = os.path.dirname(b.task_file_path("job1", "t", "stdout.txt"))
    assert not os.path.exists(os.path.join(tdir, ".container"))
    if os.geteuid() == 0 and os.path.isdir(mnt):
        for d in (mnt, mnt + "-ro", mnt + "-anon"):
            try:
                os.rmdir(d)
            except OSError:
                pass


@needs_ns
def test_keep_container_scratch_without_rm(tmp_path):
    tasks = [{"id": "t", "docker_image": "busybox", "remove_container_after_exit": False, "command": "echo keep > $TMPDIR/kept"}]
    cfg, b = make(tmp_path, tasks=tasks)
    up(cfg, b)
    run(cfg, b)
    tdir = os.path.dirname(b.task_file_path("job1", "t", "stdout.txt"))
    assert open(os.path.join(tdir, ".container", "tmp", "kept")).read().strip() == "keep"


@needs_ns
def test_restrict_default_bind_mounts_hides_node_root(tmp_path):
    tasks = [{"id": "t", "docker_image": "busybox",
              "command": 'ls "$AZ_BATCH_NODE_ROOT_DIR"; test -d "$AZ_BATCH_NODE_SHARED_DIR" && echo SHARED-VISIBLE; '
                         'test -d "$AZ_BATCH_TASK_DIR" && echo TASKDIR-VISIBLE; echo data > "$AZ_BATCH_TASK_WORKING_DIR/f"'}]
    cfg, b = make(tmp_path, tasks=tasks, job={"restrict_default_bind_mounts": True})
    up(cfg, b)
    run(cfg, b)
    out = read(b, "job1", "t")
    assert "TASKDIR-VISIBLE" in out and "SHARED-VISIBLE" not in out and "startup" not in out.split()
    assert read(b, "job1", "t", "wd/f").strip() == "data"           # what the task wrote under its own directory is real
    # without the restriction the whole node root is visible (the default bind of the reference)
    cfg2, b2 = make(tmp_path / "b", tasks=tasks)
    up(cfg2, b2)
    run(cfg2, b2)
    assert "SHARED-VISIBLE" in read(b2, "job1", "t")


@pytest.mark.skipif(os.geteuid() != 0 or MODE != "mountns", reason="user_identity switching needs root")
def test_user_identity_specific_user(tmp_path, monkeypatch):
    # pytest's base directory under /tmp is 0700 root: with the task's own /tmp the state dir is re-attached below fresh 0755 directories
    monkeypatch.setenv("SHIPYARD_SANDBOX_PRIVATE_TMP", "1")
    tasks = [{"id": "t", "docker_image": "busybox", "command": 'echo "uid=$(id -u) gid=$(id -g)"; echo mine > "$AZ_BATCH_TASK_WORKING_DIR/f"'}]
    cfg, b = make(tmp_path, tasks=tasks, job={"user_identity": {"specific_user": {"uid": 12345, "gid": 23456}}})
    os.chmod(tmp_path, 0o755)
    up(cfg, b)
    run(cfg, b)
    assert "uid=12345 gid=23456" in read(b, "job1", "t")
    st = os.stat(b.task_file_path("job1", "t", "wd/f"))
    assert (st.st_uid, st.st_gid) == (12345, 23456)


@needs_ns
def test_shm_size_is_a_private_tmpfs(tmp_path):
    tasks = [{"id": "t", "docker_image": "busybox", "shm_size": "8m",
              "command": "df -k /dev/shm | tail -1 | awk '{print \"shmkb=\" $2}'; echo x > /dev/shm/in-container-only"}]
    cfg, b = make(tmp_path, tasks=tasks)
    up(cfg, b)
    run(cfg, b)
    assert "shmkb=8192" in read(b, "job1", "t")
    assert not os.path.exists("/dev/shm/in-container-only")


def test_named_container_registry_and_coordination_cleanup(tmp_path):
    """A multi-instance coordination command that daemonises (`docker run -d` in the reference) is found by container name and
    killed by `jobs cmi` / job release; while a task runs its name is in the registry."""
    tasks = [{"id": "mi", "docker_image": "busybox", "command": "sleep 0.3; echo app",
              "multi_instance": {"num_instances": 2,
                                 "coordination_command": "(sleep 300 & echo $! >> $AZ_BATCH_NODE_SHARED_DIR/daemon.pid) >/dev/null 2>&1"}}]
    cfg, b = make(tmp_path, tasks=tasks)
    up(cfg, b)
    import pathlib
    marker = pathlib.Path(b.node_shared_dir("testpool")) / "daemon.pid"
    from batch_shipyard_b200.jobs import submit
    from batch_shipyard_b200.backend.agent import NodeAgent
    submit.add_jobs(b, cfg)
    agent = NodeAgent(b, "testpool", poll=0.02)
    assert agent.acquire()
    try:
        seen_registry = False
        cdir = runspec.containers_dir(b, "testpool")
        t0 = time.time()
        while time.time() - t0 < 30:
            agent.tick()
            if os.path.isdir(cdir) and any(f.endswith(".json") for f in os.listdir(cdir)):
                seen_registry = True
            if b.get_task("job1", "mi")["state"] == "completed":
                break
            time.sleep(0.02)
    finally:
        agent.release()
    assert b.get_task("job1", "mi")["result"] == "success" and seen_registry
    assert not any(f.endswith(".json") for f in os.listdir(cdir))         # the task's own entry is gone ...
    assert any(f.endswith(".coord") for f in os.listdir(cdir))            # ... the daemonised coordination sessions are not
    pids = [int(x) for x in marker.read_text().split()]
    assert len(pids) == 2 and all(os.path.exists(f"/proc/{p}") for p in pids)
    cleaned = b.clean_mi_containers("job1")
    assert cleaned
    time.sleep(0.3)

    def gone(p):
        try:
            with open(f"/proc/{p}/stat") as f:
                return f.read().rsplit(")", 1)[1].split()[0] == "Z"
        except OSError:
            return True
    assert all(gone(p) for p in pids)
    assert not any(f.endswith(".coord") for f in os.listdir(cdir))


def test_sandbox_off_and_spec_keys(tmp_path, monkeypatch):
    tasks = [{"id": "t", "docker_image": "busybox", "shm_size": "1g", "command": "echo mode=${SHIPYARD_SANDBOX:-off}"}]
    cfg, b = make(tmp_path, tasks=tasks, job={"restrict_default_bind_mounts": True})
    up(cfg, b)
    monkeypatch.setenv("SHIPYARD_SANDBOX_MODE", "off")
    run(cfg, b)
    assert "mode=off" in read(b, "job1", "t") and _result(b, "job1", "t")["sandbox"] == "off"
    monkeypatch.delenv("SHIPYARD_SANDBOX_MODE")
    t = b.get_task("job1", "t")
    pool, job = b.get_pool("testpool"), b.get_job("job1")
    tdir = b.task_dir("testpool", "job1", "t")
    items = dict(runspec.sandbox_items(b, pool, t, tdir, runspec.base_env(b, pool, job, "t", tdir, [])))
    assert items["sandbox"] == "auto" and items["shm_bytes"] == str(1 << 30) and items["rm"] == "1"
    assert items["restrict_root"] == b.pool_root("testpool") and items["keep"] == tdir and items["name"] == "t"
    assert runspec._size_bytes("64m") == 64 << 20 and runspec._size_bytes("512k") == 512 << 10 and runspec._size_bytes("100") == 100
