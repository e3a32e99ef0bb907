"""Every shipped recipe: configs validate through the loader, and the CPU-runnable recipe bodies train at world 2 over the stub transport."""
import json
import os
import subprocess
import sys
import uuid

import pytest

from batch_shipyard_b200.config import loader, settings as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RECIPES = sorted(d for d in os.listdir(os.path.join(ROOT, "recipes")) if os.path.isdir(os.path.join(ROOT, "recipes", d, "config")))


def test_all_reference_target_recipes_present():
    for name in ("PyTorch-GPU", "TensorFlow-Distributed", "mpiBench-OpenMPI", "HPCG-Infiniband-IntelMPI", "CNTK-GPU-OpenMPI",
                 "OSUMicroBenchmarks-Infiniband-MVAPICH", "MXNet-GPU"):
        assert name in RECIPES
        assert os.path.exists(os.path.join(ROOT, "recipes", name, "README.md"))


@pytest.mark.parametrize("recipe", RECIPES)
def test_recipe_config_validates(recipe):
    """Every config file of every recipe passes the strict schema validation; job commands point at files that exist."""
    cfg = loader.load_configs(configdir=os.path.join(ROOT, "recipes", recipe, "config"))
    if "pool_specification" in cfg:
        assert S.pool_id(cfg)
    gr = cfg.get("global_resources") or {}
    images = set(gr.get("docker_images") or []) | set(gr.get("singularity_images") or [])
    for job in cfg.get("job_specifications") or []:
        for task in job["tasks"]:
            # `jobs add` refuses a task whose image is not a global resource (unless the job opts out): the dry-run does not check this
            image = task.get("docker_image") or task.get("singularity_image")
            assert job.get("allow_run_on_missing_image") or image is None or image in images, (image, sorted(images))
            mi = task.get("multi_instance")
            if mi is not None:
                assert mi["num_instances"] == "pool_current_dedicated" and mi["mpi"]["runtime"] in ("openmpi", "mpich", "mvapich", "intelmpi", "intelmpi-ofa")
            for tok in task["command"].split():
                if tok.startswith("$SHIPYARD_HOME/"):
                    rel = tok[len("$SHIPYARD_HOME/"):]
                    assert os.path.exists(os.path.join(ROOT, rel)) or rel.startswith("batch_shipyard_b200/_native/"), rel
    if "remote_fs" in cfg:
        assert next(iter(S.remotefs_storage_clusters(cfg).values())).vm_count >= 1
    if "slurm" in cfg:
        assert S.slurm_options(cfg)["cluster_id"] == "myslurmcluster"


def test_recipe_catalogue_covers_the_reference():
    """One directory per reference recipe (the two Windows recipes under their name without the `-Windows` suffix)."""
    ref = os.path.join(ROOT, "tests", "golden", "reference", "recipes")             # the recipe catalogue of Batch Shipyard 3.9.1
    want = {d.replace("-Windows", "") for d in os.listdir(ref) if os.path.isdir(os.path.join(ref, d))}   # DiskSpd / DotNet: Linux retargets
    assert want <= set(RECIPES), sorted(want - set(RECIPES))


def _run_world(script, args, world=2, timeout=300):
    session = "rt" + uuid.uuid4().hex[:10]
    procs = []
    for r in range(world):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE=str(world), SHIPYARD_GPU="-1", SHIPYARD_COLL_SESSION=session)
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, script)] + args, env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True, cwd=ROOT))
    outs = [p.communicate(timeout=timeout)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(outs)
    line = [l for l in outs[0].splitlines() if l.startswith("{")][-1]
    return json.loads(line)


def test_quantised_gradient_recipe_world2():
    q8 = _run_world("recipes/CNTK-GPU-OpenMPI/train_quantized.py", ["-q", "8", "--epochs", "1", "--steps_per_epoch", "25", "--batch", "32"])
    q32 = _run_world("recipes/CNTK-GPU-OpenMPI/train_quantized.py", ["-q", "32", "--epochs", "1", "--steps_per_epoch", "25", "--batch", "32"])
    assert q8["world"] == 2 and q8["last_loss"] < q8["first_loss"] - 0.3
    assert abs(q8["last_loss"] - q32["last_loss"]) < 0.1            # fp8 on the wire trains like fp32 on the wire
    assert q8["wire_bytes"] < 0.27 * q32["wire_bytes"]


def test_tensorflow_distributed_recipe_world2():
    r = _run_world("recipes/TensorFlow-Distributed/mnist_replica.py", ["--train_steps", "60"])
    assert r["world"] == 2 and r["final_loss"] < 1.0 and r["transport"] == "stub"


def test_osu_recipe_runs_through_the_cli_with_osu_output(tmp_path):
    """The OSU recipe end to end on a 2-slot CPU pool: pool add, jobs add, and the task's stdout is an OSU latency table (-f columns)."""
    env = dict(os.environ, SHIPYARD_STATE_DIR=str(tmp_path / "state"), SHIPYARD_FAKE_GPUS="2")
    cfg = os.path.join(ROOT, "recipes", "OSUMicroBenchmarks-Infiniband-MVAPICH", "config")
    sh = os.path.join(ROOT, "shipyard")
    try:
        p = subprocess.run([sh, "pool", "add", "--configdir", cfg, "-y", "--raw"], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
        assert p.returncode == 0, p.stdout[-2000:]
        p = subprocess.run([sh, "jobs", "add", "--configdir", cfg, "--tail", "stdout.txt"], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
        assert p.returncode == 0, p.stdout[-3000:]
        out = p.stdout
        assert "# OSU MPI Allreduce Latency Test" in out and "Avg Latency(us)" in out and "Iterations" in out, out[-3000:]
        rows = [ln.split() for ln in out.splitlines() if ln[:1].isdigit()]
        sizes = [int(r[0]) for r in rows if len(r) == 5]
        assert sizes[0] == 4 and sizes[-1] == 1 << 20 and sizes == [4 << i for i in range(len(sizes))], sizes
        assert all(float(r[2]) <= float(r[1]) <= float(r[3]) for r in rows if len(r) == 5)
    finally:
        subprocess.run([sh, "pool", "del", "--configdir", cfg, "-y"], env=env, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, timeout=120)


@pytest.mark.parametrize("bench,header", [("pt2pt/osu_latency", "Latency (us)"), ("pt2pt/osu_bw", "Bandwidth (MB/s)"), ("collective/osu_alltoall", "Avg Latency(us)")])
def test_osu_front_end_point_to_point_and_collectives(bench, header):
    """The OSU front end on two host ranks (shared-memory transport): benchmark names with their directory prefix, -m ranges, OSU tables."""
    exe = os.path.join(ROOT, "batch_shipyard_b200", "_native", "shipyard-mpibench")
    session = "osu" + uuid.uuid4().hex[:10]
    procs = [subprocess.Popen([exe, "--osu", bench, "-m", "8:4096", "-i", "50", "-x", "5"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                              env=dict(os.environ, RANK=str(r), WORLD_SIZE="2", SHIPYARD_COLL_SESSION=session, SHIPYARD_GPU="-1")) for r in range(2)]
    outs = [p.communicate(timeout=120)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    rows = [ln.split() for ln in outs[0].splitlines() if ln[:1].isdigit()]
    assert header in outs[0] and [int(r[0]) for r in rows] == [8 << i for i in range(10)], outs[0]
    assert all(float(r[1]) > 0 for r in rows)


@pytest.mark.parametrize("recipe,key", [("HPLinpack-Infiniband-IntelMPI", "scaled_residual"), ("HPCG-Infiniband-IntelMPI", "validity")])
def test_hpc_recipes_run_through_the_cli_on_a_cpu_pool(recipe, key, tmp_path):
    """The GPU-sized HPC recipes on a 2-slot CPU pool: the bodies detect the virtual slots, downscale (and say so) and still pass their
    validity checks; exit code 0 through pool add / jobs add.  The ranks see no CUDA device, also on a machine that has one."""
    env = dict(os.environ, SHIPYARD_STATE_DIR=str(tmp_path / "state"), SHIPYARD_FAKE_GPUS="2", CUDA_VISIBLE_DEVICES="")
    cfg = os.path.join(ROOT, "recipes", recipe, "config")
    sh = os.path.join(ROOT, "shipyard")
    try:
        p = subprocess.run([sh, "pool", "add", "--configdir", cfg, "-y", "--raw"], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
        assert p.returncode == 0, p.stdout[-2000:]
        p = subprocess.run([sh, "jobs", "add", "--configdir", cfg, "--tail", "stdout.txt"], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
        assert p.returncode == 0 and "task_state: completed" in p.stdout and "exit_code:" not in p.stdout, p.stdout[-3000:]
        line = next(ln for ln in p.stdout.splitlines() if ln.startswith("{") and key in ln)
        out = json.loads(line)
        assert out["world"] == 2 and "downscaled_for_cpu" in out and out["transport"] == "stub", out
        assert out.get("passed", True) and (out.get("validity") or {"passed": True})["passed"], out
    finally:
        subprocess.run([sh, "pool", "del", "--configdir", cfg, "-y"], env=env, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, timeout=120)


@pytest.mark.parametrize("model,steps,lr", [("lenet", "120", "0.01"), ("resnet20", "50", "0.05")])
def test_small_model_recipe_bodies_learn(model, steps, lr):
    """The MNIST LeNet / CIFAR ResNet-20 bodies of the single-framework CPU recipes at world 2 (stub transport): the loss falls by a factor
    of four at least and the held-out synthetic images are classified."""
    script = os.path.join(ROOT, "recipes", "PyTorch-GPU", "train_resnet50.py")
    session = model + uuid.uuid4().hex[:10]
    procs = [subprocess.Popen([sys.executable, script, "--model", model, "--steps", steps, "--batch", "64", "--lr", lr], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True,
                              env=dict(os.environ, RANK=str(r), WORLD_SIZE="2", SHIPYARD_COLL_SESSION=session, SHIPYARD_GPU="-1", OMP_NUM_THREADS="2"))
             for r in range(2)]
    outs = [p.communicate(timeout=600)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    out = json.loads(outs[0].strip().splitlines()[-1])
    assert out["model"] == model and out["world"] == 2 and out["last_loss"] < 0.25 * out["first_loss"] and out["test_accuracy"] > 0.9, out
