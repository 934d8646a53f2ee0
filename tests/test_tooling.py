"""Launcher / tracker / lint / baseline-arm tests (CPU only)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tracker"))


def test_lint_clean():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "lint.py")], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:]


def test_tracker_topology():
    import tracker

    for n in (1, 2, 5, 8, 13):
        tree, parent, ring = tracker.link_map(n)
        assert sorted(tree) == list(range(n))
        assert parent[0] == -1
        # ring is a single cycle 0 -> 1 -> ... -> n-1 -> 0 after relabelling
        for r in range(n):
            assert ring[r] == ((r - 1) % n, (r + 1) % n)
        # tree edges are symmetric and connect everything
        for r, nbrs in tree.items():
            for x in nbrs:
                assert r in tree[x]
        seen, stack = {0}, [0]
        while stack:
            for x in tree[stack.pop()]:
                if x not in seen:
                    seen.add(x)
                    stack.append(x)
        assert len(seen) == n


def test_dmlc_local_launcher(built_native_tree):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tracker", "dmlc_local.py"), "-n", "2", "-s", "2",
                        os.path.join(built_native_tree, "test_kv_app"), "300", "2", "2"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT)
    out = r.stdout + r.stderr
    assert r.returncode == 0 and out.count("test_kv_app PASSED") == 2, out[-3000:]


def test_dmlc_ssh_and_mpi_dry_run(tmp_path):
    hosts = tmp_path / "hosts"
    hosts.write_text("nodeA:2200\n# comment\nnodeB\n")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tracker", "dmlc_ssh.py"), "-n", "2", "-s", "1",
                        "-H", str(hosts), "--dry-run", "echo", "hi"], capture_output=True, text=True)
    assert r.returncode == 0
    lines = [line for line in r.stdout.splitlines() if line.startswith("ssh ")]
    assert len(lines) == 3 and "nodeA -p 2200" in lines[0] and "DMLC_ROLE=server" in lines[0]
    assert "DMLC_ROLE=worker" in lines[1] and "nodeB -p 22" in lines[1]
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tracker", "dmlc_mpi.py"), "-n", "4", "-s", "2",
                        "--dry-run", "./app"], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.count("mpirun -n") == 2


def test_reference_arm_runs_unmodified_reference():
    """bench.py --impl reference builds baseline/_ref and runs the reference's own test_benchmark.
    tests/golden/reference_test_benchmark_worker.log is the worker's output of one run of the unmodified
    reference with the arguments below (ZMQ van, 1 worker + 1 server): the arm must read the goodput of
    its last window from it. The live run follows where the reference's sources are at hand."""
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    import bench
    import build_reference

    with open(os.path.join(ROOT, "tests", "golden", "reference_test_benchmark_worker.log")) as f:
        assert bench.reference_goodput(f.read()) == 11.8584
    assert bench.reference_goodput("Start ZMQ recv thread\n") is None
    if not os.path.isdir(build_reference.REF_SRC) and not os.path.isdir(os.path.join(build_reference.DST, "src")):
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "4",
                        "--warmup", "1", "--len", "256000", "--keys-per-server", "4"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference"
    assert "unavailable" in line or line["value"] > 0


REQUIRED_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                 "scaling", "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches"}


@pytest.mark.parametrize("extra", [["--e2e-native", "--fused-pushpull"],
                                   ["--metric", "llama", "--model", "tiny", "--seq-len", "64"],
                                   ["--metric", "resnet", "--model", "tiny", "--image-batch", "2"]])
def test_bench_script_control_flow_on_cpu(extra, tmp_path):
    """bench.py --device cpu walks the same code as a GPU run (warm-up, timed region, end-to-end
    pass, JSON line) over the shm van and the host engine: a typo in the script must not wait for
    the round-end GPU run to be found. The numbers it prints are not benchmark results."""
    import numpy as np

    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--device", "cpu", "--steps", "3", "--warmup", "3",
           "--len", "65536", "--keys-per-server", "4", "--sweep", "4096", "--dump-outputs", str(tmp_path), *extra]
    env = dict(os.environ, PSLITE_NO_AUTOBUILD="1", CUDA_VISIBLE_DEVICES="")
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert REQUIRED_KEYS <= set(line), REQUIRED_KEYS - set(line)
    assert line["value"] > 0 and line["e2e"]["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["d2h_bytes_per_step"] > 0
    if "--e2e-native" in extra:
        assert line["e2e"]["native_call"]["value"] > 0 and line["fused_pushpull"]["value"] > 0
    dumped = {p.stem: np.load(p) for p in tmp_path.glob("*.npy")}
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in dumped.values()), dumped
    if "--metric" in extra:
        assert set(dumped) == {"loss", "parameters"} and dumped["loss"].shape == (1,)
        assert dumped["parameters"].size > 0 and dumped["parameters"].any()
    else:  # every byte the last timed round pulled back: the constant the benchmark pushes
        assert set(dumped) == {"pulled_values"} and dumped["pulled_values"].size == 4 * 65536
        assert (dumped["pulled_values"] == 1).all()


def test_bench_dump_outputs_samples_large_outputs(tmp_path):
    """past the size limit --dump-outputs keeps a seeded sample of every array, at the same positions in
    every run, and never drops a one-element output such as a loss"""
    import numpy as np
    import torch

    sys.path.insert(0, ROOT)
    import bench

    n = bench.DUMP_MAX_ELEMS
    arrays = {"x": [torch.arange(n, dtype=torch.int32), torch.arange(7, dtype=torch.int32)],
              "loss": [torch.tensor(2.5)]}
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays)
    a, b = (np.load(tmp_path / run / "x.npy") for run in ("a", "b"))
    assert a.dtype == np.float32 and np.array_equal(a, b)
    assert 0.99 * n < a.size and a.size + 1 <= n and len(np.unique(a)) < a.size  # a sample, not the whole
    assert (np.diff(a[:-6]) >= 0).all() and a[-6:].max() < 7
    assert np.load(tmp_path / "a" / "loss.npy").tolist() == [2.5]
    assert sum(os.path.getsize(p) for p in (tmp_path / "a").iterdir()) <= 64 << 20
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs",
                        str(tmp_path / "c")], capture_output=True, text=True, timeout=60, cwd=ROOT)
    assert r.returncode != 0 and "--dump-outputs" in r.stderr and not (tmp_path / "c").exists()


def test_bench_script_multi_process_on_cpu():
    """the torchrun form the driver uses for N > 1: N workers + N servers, one of each per rank (the
    same topology at every N); --topology split gives N/2 + N/2"""
    from pslite_b200.utils.env import free_port

    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=4", "--master-addr",
           "127.0.0.1", "--master-port", str(free_port()), os.path.join(ROOT, "bench.py"), "--device", "cpu",
           "--gpus", "4", "--steps", "3", "--warmup", "3", "--len", "65536", "--keys-per-server", "4", "--e2e-native"]
    env = dict(os.environ, PSLITE_NO_AUTOBUILD="1", CUDA_VISIBLE_DEVICES="", OMP_NUM_THREADS="1")
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
    line = json.loads([l for l in r.stdout.strip().splitlines() if l.startswith("{")][-1])
    assert line["n_gpus"] == 4 and line["config"]["num_workers"] == 4 and line["config"]["num_servers"] == 4
    assert line["value"] > 0 and line["e2e"]["value"] > 0 and "roofline" in line
    cmd = cmd[:-1] + ["--topology", "split", "--no-e2e"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
    line = json.loads([l for l in r.stdout.strip().splitlines() if l.startswith("{")][-1])
    assert line["config"]["num_workers"] == 2 and line["config"]["num_servers"] == 2 and line["value"] > 0


def test_bench_script_across_hosts_on_cpu():
    """two ranks that take each other for different hosts: half of the keys move one-sidedly (own server),
    the other half in socket frames with the values staged through the host; bench.py's own data check
    (every pulled byte compared with what was pushed) must hold on both halves"""
    from pslite_b200.utils.env import free_port

    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", str(free_port()), os.path.join(ROOT, "bench.py"), "--device", "cpu",
           "--gpus", "2", "--steps", "3", "--warmup", "3", "--len", "65536", "--keys-per-server", "4"]
    env = dict(os.environ, PSLITE_NO_AUTOBUILD="1", CUDA_VISIBLE_DEVICES="", OMP_NUM_THREADS="1",
               PS_TEST_HOST_PER_RANK="1", PS_TEST_STAGE_ARENA="1")
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
    line = json.loads([l for l in r.stdout.strip().splitlines() if l.startswith("{")][-1])
    stats = line["van_stats_rank0"]["worker"]
    assert stats["staged_copies"] > 0 and stats["onesided_copies"] > 0, stats
    assert line["value"] > 0 and line["e2e"]["value"] > 0


def test_native_initialises_torch_first():
    """the extension hands tensors to Python: loading it without the torch package crashed later"""
    code = "import sys; import pslite_b200; pslite_b200.native(); assert 'torch' in sys.modules; print('ok')"
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=ROOT,
                       env=dict(os.environ, PSLITE_NO_AUTOBUILD="1", CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0 and "ok" in r.stdout, (r.stdout + r.stderr)[-2000:]


def test_scheduler_child_dies_with_a_crashed_launcher():
    """init_ps spawns the scheduler; if the launching process dies without cleanup the scheduler
    must not stay behind (it would hold the port and the launcher's output pipe)"""
    import time

    code = ("import os, sys; sys.path.insert(0, %r)\n"
            "import pslite_b200\n"
            "from pslite_b200.parallel.launch import init_ps\n"
            "pslite_b200.native()\n"
            "ctx = init_ps('joint', van='shm')\n"
            "print('SCHED', ctx.scheduler.pid, flush=True)\n"
            "os._exit(3)\n" % ROOT)
    r = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
                       timeout=300, cwd=ROOT, env=dict(os.environ, PSLITE_NO_AUTOBUILD="1", CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 3
    pid = int([l for l in r.stdout.splitlines() if l.startswith("SCHED")][0].split()[1])
    for _ in range(100):
        if not os.path.exists(f"/proc/{pid}"):
            break
        try:  # a zombie whose parent is gone is reaped by init; "Z" counts as gone
            if open(f"/proc/{pid}/stat").read().split(")")[1].split()[0] == "Z":
                break
        except OSError:
            break
        time.sleep(0.1)
    else:
        os.kill(pid, 15)
        raise AssertionError(f"scheduler {pid} outlived its launcher")


# what a copy of the built tree for a GPU machine leaves out: history, caches, sanitizer builds, profiler reports
SNAPSHOT_SKIP_DIRS = {".git", "build-asan", "build-tsan", ".tmp", "__pycache__", ".pytest_cache", ".hypothesis"}
SNAPSHOT_SKIP_FILES = ["*.pyc", "*.ncu-rep"]


def _snapshot_bytes(root):
    """Size of the built tree without SNAPSHOT_SKIP_DIRS and SNAPSHOT_SKIP_FILES."""
    import fnmatch

    dir_rules, file_rules = SNAPSHOT_SKIP_DIRS, SNAPSHOT_SKIP_FILES
    total, biggest = 0, []
    for dirpath, dirnames, filenames in os.walk(root):
        rel = os.path.relpath(dirpath, root)
        dirnames[:] = [d for d in dirnames if d not in dir_rules
                       and os.path.normpath(os.path.join(rel, d)) not in dir_rules]
        for f in filenames:
            if any(fnmatch.fnmatch(f, r) for r in file_rules):
                continue
            p = os.path.join(dirpath, f)
            if os.path.islink(p):
                continue
            n = os.path.getsize(p)
            total += n
            biggest.append((n, os.path.relpath(p, root)))
    return total, sorted(biggest, reverse=True)[:8]


def test_snapshot_under_256MiB():
    """The built tree must stay small enough to copy to a GPU machine: a default build once carried 691 MB of
    DWARF."""
    total, biggest = _snapshot_bytes(ROOT)
    assert total < 256 << 20, f"snapshot {total >> 20} MiB; biggest: {biggest}"
    mk = open(os.path.join(ROOT, "Makefile")).read()
    flags = [ln for ln in mk.splitlines() if ln.startswith("CXXFLAGS :=")][0]
    assert " -g" not in flags, "default CXXFLAGS must not carry DWARF (use DEBUG=1)"
