"""bench.py contract checks that do not need a GPU: the reference (CPU) arm prints exactly one JSON line with the keys
the driver reads, and the own arm refuses to run without a GPU instead of falling back.  The checks of --dump-outputs
that run the own arm need a GPU (-m gpu), the sharded one at least two."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bench_module():
    """bench.py imported for its constants.  Importing it sets the CPU arm's OpenMP variables (OMP_PROC_BIND, ...) in
    os.environ; the environment is restored so that processes later tests start do not inherit them."""
    saved = dict(os.environ)
    try:
        import bench
    finally:
        os.environ.clear()
        os.environ.update(saved)
    return bench


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "1"], cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "Gkeys/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["gpu_launches"] == 0


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                       cwd=ROOT, capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_own_arm_needs_a_gpu():
    import torch

    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, "bench.py", "--steps", "1", "--warmup", "1"], cwd=ROOT, capture_output=True,
                       text=True, timeout=300)
    assert r.returncode != 0 and r.stdout.strip() == ""  # no number is ever produced by a CPU path


def test_both_arms_print_the_same_metric_and_workload_strings(bench_module):
    """The driver divides the two arms' values only if metric/unit/config agree: both lines are built from the same
    constants (round 1 printed two different metric strings and got no ratio)."""
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert src.count('"metric": METRIC') == 2 and src.count('"workload": workload(') == 2
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                       cwd=ROOT, capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, RANK="0", WORLD_SIZE="2", LOCAL_RANK="0", OMP_NUM_THREADS="1"))
    d = json.loads(r.stdout.strip())
    bench = bench_module
    assert d["metric"] == bench.METRIC and d["config"]["workload"] == bench.workload(bench.LOG2_N, 2)
    # torchrun exports OMP_NUM_THREADS=1: the CPU leg must still use every physical core it may run on
    assert d["cpu_baseline"]["cores"] == bench.HOST_THREADS >= 1


def test_gpu_arm_under_torchrun_does_not_pin_its_main_thread():
    """Round 2's N = 4 / 8 scaling regression: bench.py exported OMP_PROC_BIND in every rank, the OpenMP runtime then pinned
    every rank's main thread to core 0, and the ranks time-shared one core.  A rank of the GPU arm (WORLD_SIZE > 1, no
    --impl reference) must keep the launcher's OMP settings and its affinity mask; the CPU arm keeps the binding."""
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import os,sys; sys.argv=['bench.py'{extra}]; os.environ['WORLD_SIZE']='4'; os.environ['RANK']='1'; "
            "os.environ['OMP_NUM_THREADS']='1'; os.environ.pop('OMP_PROC_BIND', None); os.environ.pop('OMP_PLACES', None); before=len(os.sched_getaffinity(0)); "
            "import importlib.util as u; s=u.spec_from_file_location('bench', os.path.join(r'" + root + "', 'bench.py')); "
            "m=u.module_from_spec(s); s.loader.exec_module(m); import torch; "
            "print(before, len(os.sched_getaffinity(0)), os.environ.get('OMP_PROC_BIND'), os.environ['OMP_NUM_THREADS'])")
    out = subprocess.run([sys.executable, "-c", code.format(extra=",'--gpus','4'")], capture_output=True, text=True, timeout=300)
    before, after, bind, threads = out.stdout.split()
    assert before == after and bind == "None" and threads == "1", out.stdout + out.stderr
    out = subprocess.run([sys.executable, "-c", code.format(extra=",'--impl','reference'")], capture_output=True, text=True, timeout=300)
    assert out.stdout.split()[2] == "spread", out.stdout + out.stderr


def test_dump_outputs_and_steps_arguments_are_checked():
    for extra in (["--steps", "0"], ["--dump-outputs"]):  # no timed step; no directory
        r = subprocess.run([sys.executable, "bench.py", *extra], cwd=ROOT, capture_output=True, text=True, timeout=300)
        assert r.returncode == 2 and r.stdout.strip() == "", r.stderr


def _sample(want, bench):
    """want at the positions bench.py --dump-outputs keeps (all of them when there are no more than bench.DUMP_SAMPLE)."""
    import numpy as np

    if want.size > bench.DUMP_SAMPLE:
        want = want[np.sort(np.random.default_rng(bench.SEED).choice(want.size, size=bench.DUMP_SAMPLE, replace=False))]
    return want.astype(np.float64)


def test_reference_arm_dumps_its_sorted_sample(tmp_path, oracle, bench_module):
    """--impl reference --dump-outputs: the CPU arm's last timed sort of its 2^CPU_SAMPLE_LOG2-key sample."""
    import numpy as np

    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--dump-outputs", str(tmp_path)], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    got = np.load(tmp_path / "sorted_keys.npy")
    want = oracle.init_random_u32(1 << bench_module.CPU_SAMPLE_LOG2, 0, bench_module.SEED)
    assert oracle.sort_parallel_inplace(want) == 0
    assert got.dtype == np.float64 and np.array_equal(got, _sample(want, bench_module))


@pytest.mark.gpu
def test_dump_outputs_writes_the_sorted_sample(tmp_path, oracle, bench_module):
    """--dump-outputs: the last timed step's sorted keys at the seeded sample positions, equal to the oracle's sort; and
    --steps sets the number of timed sorts, counted by the sorter's pass counter (gpu_launches)."""
    import numpy as np

    import gpusorting_b200 as g

    log2n, steps = 24, 2
    r = subprocess.run([sys.executable, "bench.py", "--log2n", str(log2n), "--steps", str(steps), "--no-extra",
                        "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], cwd=ROOT, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr
    d = json.loads(r.stdout)
    with g.OneSweepSorter(1 << log2n, 4, 0) as s:
        assert d["steps"] == steps and d["gpu_launches"] == steps * s.info("launches_per_sort")
    got = np.load(tmp_path / "sorted_keys.npy")
    want = oracle.sort_keys(oracle.init_random_u32(1 << log2n, 0, bench_module.SEED))
    assert got.dtype == np.float64 and got.size == bench_module.DUMP_SAMPLE
    assert np.array_equal(got, _sample(want, bench_module))


@pytest.mark.gpu
def test_sharded_dump_outputs_are_the_global_order(tmp_path, oracle, bench_module):
    """--dump-outputs under torchrun: every rank writes its slice of the global order; at 2^18 keys per rank every slice
    fits the per-rank sample, so the slices in rank order are the sort of all ranks' inputs (seed SEED + rank)."""
    import numpy as np
    import torch

    world = min(torch.cuda.device_count(), 4)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    log2n = 18
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node", str(world),
                        "bench.py", "--gpus", str(world), "--log2n", str(log2n), "--steps", "2",
                        "--dump-outputs", str(tmp_path)], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert json.loads(r.stdout.strip().splitlines()[-1])["n_gpus"] == world
    slices = [np.load(tmp_path / f"sorted_keys_rank{q}.npy") for q in range(world)]
    assert all(sl.size <= bench_module.DUMP_SAMPLE // world for sl in slices)
    keys = np.concatenate([oracle.init_random_u32(1 << log2n, 0, bench_module.SEED + q) for q in range(world)])
    assert np.array_equal(np.concatenate(slices), np.sort(keys).astype(np.float64))
