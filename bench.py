#!/usr/bin/env python
"""bench.py -- the contract benchmark of the OneSweep path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is ONE pass of the hot path over one batch of synthetic input: one OneSweep sort of 2^30 uint32 keys
(BASELINE.json configs[1]) per GPU, inputs already resident in HBM.  Prints ONE JSON line (rank 0).

  value / ms_per_step   whole-job Gkeys/s, device time of the sort (CUDA events on the launching stream, max over
                        ranks); the unsorted input is restored by an untimed device copy between steps
  roofline              the dominant kernel (one DigitBinningPass): 8 B/key algorithmic bytes per launch divided by
                        its CUDA-event duration measured live in the timed steps, against MEASURED_PEAKS.json
  e2e                   same metric through the C-ABI host-buffer call (pinned host memory in, sorted data back out:
                        H2D + sort + D2H inside the timed region)
  cpu_baseline          the oracle's host-parallel port of the same algorithm (and std::sort) on the box's host cores,
                        on a bounded sample; reported, not the target
  --impl reference      the reference has no CPU implementation of this path (SURVEY D2): this arm times the oracle's
                        host-parallel OneSweep port on all host threads on a bounded sample of the same workload
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

def _physical_cores() -> int:
    """Physical cores this process may run on (affinity mask, one per SMT sibling set)."""
    try:
        cpus = sorted(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1
    seen = set()
    for c in cpus:
        try:
            sib = open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list").read().strip()
        except OSError:
            sib = str(c)
        seen.add(sib)
    return max(1, len(seen))


HOST_THREADS = _physical_cores()
# The CPU legs use every physical core, whatever the launcher exported (torchrun sets OMP_NUM_THREADS=1).  Must happen
# before numpy / torch / the oracle load an OpenMP runtime.  ONLY for processes that run a CPU leg (the single-GPU arm's
# cpu_baseline, the --impl reference arm): OMP_PROC_BIND pins the MAIN thread of the process to the first place as soon as
# the OpenMP runtime loads, i.e. with N ranks on a box all N main threads land on core 0 and time-share it.  Round 2 found
# that the hard way: with the binding set in every rank the sharded step took 30 / 77 ms at N = 4 / 8 instead of 17 / 18
# (profiles/r02_sharded_host_wait.txt) -- the rank whose busy-polling thread had run longest was descheduled and reacted
# to its GPU ~10 ms late, at every collective.
_WORLD = int(os.environ.get("WORLD_SIZE", "1"))
_CPU_ARM = "reference" in sys.argv[1:]
if _WORLD == 1 or _CPU_ARM:
    os.environ["OMP_NUM_THREADS"] = str(HOST_THREADS)
    os.environ.setdefault("OMP_PROC_BIND", "spread")
    os.environ.setdefault("OMP_PLACES", "cores")

LOG2_N = 30            # BASELINE.json configs[1]: 2^30 uint32 keys-only, uniform random, 1xB200
METRIC = "OneSweep sort throughput, 2^30 uint32 keys per GPU, keys-only, uniform-random"  # both arms print this string
DATA = "synthetic (reference InitRandom generator, seed 10, entropy preset 1)"


def workload(log2n: int, world: int) -> str:
    w = f"2^{log2n} uint32 keys-only OneSweep per GPU, uniform-random (BASELINE.json configs[1])"
    return w if world == 1 else w + f"; {world} GPUs: MSD bucket exchange over NVLink then local OneSweep"

SEED = 10              # the reference's benchmark seed (GPUSortingCUDA.cu:22)
CPU_SAMPLE_LOG2 = 27   # bounded CPU sample of the same workload (1/8 of it)
ALG_BYTES_PER_KEY_PER_PASS = 8  # SURVEY 8(d): one DigitBinningPass reads 4 B and writes 4 B per key
DUMP_SAMPLE = 1 << 22  # --dump-outputs: values kept per output array


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic_bytes():
    """dram read+write bytes per launch of the dominant kernel from the committed ncu capture (profiles/)."""
    p = os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return d
        except Exception:
            pass
    return None


# NVML queries take driver locks that CUDA API calls of the same process also need, and the sampling thread competes for the
# GIL: at 2 ms per sample the sharded loop (which has a host sync per step) lost ~5 ms per step on the sampled rank
# (profiles/r02_bench_n2_sampler_2ms.json).  20 ms still gives >= 10 samples inside the shortest timed region.
CLOCK_SAMPLE_S = float(os.environ.get("OSB_CLOCK_SAMPLE_MS", "20")) / 1e3


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksEventReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksEventReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksEventReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksEventReasonSwPowerCap: "sw_power_cap",
            nv.nvmlClocksEventReasonHwPowerBrakeSlowdown: "hw_power_brake",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(CLOCK_SAMPLE_S)

    def result(self):
        self.stop_flag = True
        if self.nv is None or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


def _cpu_sort_sample(steps: int, warmup: int):
    """The CPU leg shared by cpu_baseline and --impl reference: the oracle's host-parallel OneSweep port on
    HOST_THREADS threads over a 2^CPU_SAMPLE_LOG2-key sample of the workload.  Returns (best_s, mean_s, all_s, orc, src, work),
    work holding the last timed step's sorted keys."""
    from tests import oraclelib
    import numpy as np

    orc = oraclelib.load_oracle()
    n = 1 << CPU_SAMPLE_LOG2
    src = orc.init_random_u32(n, 0, SEED)
    work = src.copy()
    alt = np.zeros_like(src)  # pre-faulted scratch: page faults are not part of the sort
    for _ in range(max(warmup, 1)):
        np.copyto(work, src)
        orc.sort_parallel_inplace(work, threads=HOST_THREADS, alt=alt)
    times = []
    for _ in range(max(steps, 1)):
        np.copyto(work, src)
        t0 = time.perf_counter()
        orc.sort_parallel_inplace(work, threads=HOST_THREADS, alt=alt)
        times.append(time.perf_counter() - t0)
    assert orc.validate(work) == 0
    return min(times), sum(times) / len(times), times, orc, src, work


def _sample_text(kind: str) -> str:
    return (f"2^{CPU_SAMPLE_LOG2} of the 2^{LOG2_N} uint32 keys (1/{1 << (LOG2_N - CPU_SAMPLE_LOG2)} of the workload, InitRandom "
            f"seed {SEED}) per step; host-parallel 4-pass LSD radix port of OneSweep (oracle/oracle.c orc_onesweep_parallel) "
            f"on {HOST_THREADS} threads = physical cores of the affinity mask, OMP_PROC_BIND={os.environ.get('OMP_PROC_BIND')}; {kind}")


def cpu_baseline():
    """Bounded CPU sample: the oracle's host-parallel OneSweep port on all physical cores + std::sort on one core."""
    import numpy as np

    best, mean, times, orc, src, _ = _cpu_sort_sample(steps=5, warmup=1)
    n = src.size
    m = 1 << 24
    w2 = src[:m].copy()
    t0 = time.perf_counter()
    orc.lib.orc_std_sort_u32(w2.ctypes.data, m)
    std_dt = time.perf_counter() - t0
    work = src.copy()
    t0 = time.perf_counter()
    orc.lib.orc_parallel_sort_u32(work.ctypes.data, n, HOST_THREADS)  # libstdc++ parallel-mode std::sort, all cores
    par_dt = time.perf_counter() - t0
    return {
        "value": round(n / best / 1e9, 4), "unit": "Gkeys/s", "cores": HOST_THREADS, "kind": "port",
        "sample": _sample_text("best of 5"), "mean_gkeys_s": round(n / mean / 1e9, 4),
        "std_sort_1_thread_gkeys_s": round(m / std_dt / 1e9, 4), "std_sort_sample": "2^24 keys, std::sort, 1 thread",
        "gnu_parallel_sort_gkeys_s": round(n / par_dt / 1e9, 4),
        "gnu_parallel_sort_sample": f"2^{CPU_SAMPLE_LOG2} keys, __gnu_parallel::sort, {HOST_THREADS} threads",
    }


def run_reference_arm(args, rank, world, emit):
    """--impl reference: the CPU leg (rank 0 only; other ranks exit 0 without work).  The reference has no CPU
    implementation of this path (SURVEY D2) and its CUDA kernels are not a CPU arm, so this times the oracle's
    host-parallel port of the same algorithm.  value = best of the K timed steps (the most favourable number for the
    CPU side; the mean is reported beside it)."""
    if rank != 0:
        return
    best, mean, times, orc, src, work = _cpu_sort_sample(steps=args.steps, warmup=args.warmup)
    if args.dump_outputs:
        import numpy as np
        import torch

        dump_outputs(args.dump_outputs, {"sorted_keys": torch.from_numpy(work.view(np.int32))})
    n = src.size
    value = n / best / 1e9
    line = {
        "impl": "reference", "metric": METRIC,
        "value": round(value, 4), "unit": "Gkeys/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(best * 1e3, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32",
        "data": DATA,
        "config": {"workload": workload(LOG2_N, max(args.gpus, 1)),
                   "cpu_sample": _sample_text(f"value = best of {args.steps} timed steps"),
                   "mean_gkeys_s": round(n / mean / 1e9, 4), "ms_per_step_mean": round(mean * 1e3, 3),
                   "note": "the reference has no CPU implementation of this path (SURVEY D2); this is the oracle port"},
        "cpu_baseline": {"value": round(value, 4), "unit": "Gkeys/s", "cores": HOST_THREADS, "kind": "port",
                         "sample": _sample_text(f"best of {args.steps} timed steps")},
        "e2e": {"value": round(value, 4), "unit": "Gkeys/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def main():
    # stdout carries exactly ONE JSON line: libraries that print to fd 1 (e.g. the NCCL version banner) go to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log2n", type=int, default=LOG2_N, help="keys per GPU (development only; the contract is 30)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip extra_configs (pairs, u64) and ref_cuda (development)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the sorted keys of the last one to DIR/sorted_keys.npy (float64; "
                         f"a fixed seeded sample of {DUMP_SAMPLE} positions when the output is larger), so that two builds "
                         "can be compared output for output.  With N > 1 GPUs every rank writes its slice of the global "
                         f"order to DIR/sorted_keys_rank<r>.npy, sampled to {DUMP_SAMPLE} / N positions")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "ours" and args.warmup < 3:
        print(f"bench.py: --warmup {args.warmup} raised to 3 (timing rule: W >= 3)", file=sys.stderr)
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world, emit)
        return

    import torch
    import torch.distributed as dist

    import gpusorting_b200 as g  # raises if the CUDA library is missing: there is no fallback

    assert torch.cuda.is_available(), "bench.py (ours) needs a GPU"
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    n = 1 << args.log2n
    peak, peak_src = measured_peak_gbs()

    if world > 1:
        from gpusorting_b200 import sharded

        result = sharded.bench_sharded(args, rank, world, local_rank, n)
    else:
        result = bench_single(args, g, n, local_rank)

    # max over ranks of the device time
    ms = result["ms_per_step"]
    e2e_ms = result["e2e_ms_per_step"]
    if world > 1:
        t = torch.tensor([ms, e2e_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms = float(t[0]), float(t[1])
    total_keys = n * world
    value = total_keys / (ms / 1e3) / 1e9
    e2e_value = total_keys / (e2e_ms / 1e3) / 1e9

    if rank == 0:
        pass_ms = result["pass_ms"]
        achieved = ALG_BYTES_PER_KEY_PER_PASS * n / (pass_ms / 1e3) / 1e9
        traffic = ncu_traffic_bytes()
        # dram read+write bytes of ONE launch of the dominant kernel from the committed `ncu --set full` capture; used
        # as measured only when the capture was taken at this n, otherwise it is not reported as a measurement
        traffic_bytes, traffic_note = None, "no ncu capture committed for this kernel yet"
        if traffic:
            traffic_note = traffic.get("note", "")
            if int(traffic.get("log2n", -1)) == args.log2n and "dram_bytes_per_launch" in traffic:
                traffic_bytes = int(traffic["dram_bytes_per_launch"])
            else:
                traffic_note = (f"capture is at 2^{traffic.get('log2n')} (traffic/algorithmic = "
                                f"{traffic.get('traffic_over_algorithmic')}), not at this n: not reported as measured. " + traffic_note)
        line = {
            "metric": METRIC,
            "value": round(value, 3), "unit": "Gkeys/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(ms, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32", "data": DATA,
            "config": {
                "workload": workload(args.log2n, world),
                "keys_per_gpu": n, "total_keys": total_keys, "passes": 4, "digit_bits": 8,
                "variant": result["variant"], "tile_keys": result["tile_keys"], "rank_mode": result["rank_mode"],
                "timing": "CUDA events on the launching stream around each sort, summed over the K steps, max over ranks; "
                          "unsorted input restored by an untimed device copy between steps",
                "l2": "inputs (4 GiB) are larger than L2 (126 MB)",
                "roofline_pct_of_peak_32B_per_key": round(32.0 * total_keys / world / (ms / 1e3) / 1e9 / peak * 100, 2),
            },
            "roofline": {
                "bound": "hbm", "kernel": result["kernel"], "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 4),
                "traffic": traffic_bytes,
                "traffic_note": traffic_note,
                "algorithmic_bytes_per_launch": ALG_BYTES_PER_KEY_PER_PASS * n,
                "launch_ms": round(pass_ms, 4), "peak_source": peak_src,
                "kernel_ms": {k: round(v, 4) for k, v in result["kernel_ms"].items()},
            },
            "e2e": {"value": round(e2e_value, 3), "unit": "Gkeys/s", "ms_per_step": round(e2e_ms, 3),
                    "steps": result["e2e_steps"], "h2d_bytes_per_step": result["h2d_bytes"],
                    "d2h_bytes_per_step": result["d2h_bytes"],
                    "api": result.get("e2e_api", "osb200_sort_host_keys_u32 (C-ABI, pinned host buffers)")},
            "gpu_launches": result["gpu_launches"],
            "clocks": result["clocks"],
            "verified": result["verified"],
        }
        for k in ("extra_configs", "ref_cuda", "entropy_sweep", "phases_ms", "per_rank"):
            if k in result:
                line[k] = result[k]
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline()
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def multiset_checksum(t):
    """Order-independent checksum of a device tensor's 32-bit words (sum and a mixed sum, mod 2^64), chunked."""
    import torch

    a = b = 0
    flat = t.view(torch.int32)
    step = 1 << 27
    for i in range(0, flat.numel(), step):
        x = flat[i:i + step].to(torch.int64) & 0xFFFFFFFF
        a += int(x.sum().item())
        b += int(((x * 2654435761) ^ (x >> 7)).sum().item())
    m = (1 << 64) - 1
    return a & m, b & m


def dump_outputs(out_dir, arrays, sample=DUMP_SAMPLE):
    """Writes each tensor of 32-bit unsigned words as out_dir/<name>.npy in float64 (exact for 32-bit values).  A tensor
    longer than `sample` is sampled at `sample` distinct positions drawn with seed SEED and kept in ascending order, the
    same positions on every run with the same arguments; DUMP_SAMPLE float64 values are 32 MiB."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        flat = t.reshape(-1)
        if flat.numel() > sample:
            idx = np.sort(np.random.default_rng(SEED).choice(flat.numel(), size=sample, replace=False))
            flat = flat[torch.from_numpy(idx).to(flat.device)]
        vals = flat.to(torch.int64).cpu().numpy() & 0xFFFFFFFF
        np.save(os.path.join(out_dir, f"{name}.npy"), vals.astype(np.float64))


def _time_sorts(steps, warmup, restore, sort, stream):
    """K device-timed sorts (CUDA events on the launching stream around each sort; restore() is untimed)."""
    import torch

    for _ in range(warmup):
        restore()
        sort()
    torch.cuda.synchronize()
    ev = []
    for _ in range(steps):
        restore()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        sort()
        b.record(stream)
        ev.append((a, b))
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in ev) / steps


def extra_config_pairs(g, n, peak, steps=5, warmup=3):
    """BASELINE.json configs[2]: 2^30 (uint32 key, uint32 payload) pairs, device-timed, with its own roofline."""
    import numpy as np
    import torch

    k0 = torch.empty(n, dtype=torch.int32, device="cuda")
    v0 = torch.empty(n, dtype=torch.int32, device="cuda")
    g.init_random(k0, 0, SEED, payload=v0, payload_is_index=True)
    k, v = torch.empty_like(k0), torch.empty_like(v0)
    s = g.OneSweepSorter(n, 4, 4)
    s.set_option("profile", 1)
    stream = torch.cuda.current_stream()
    ck = multiset_checksum(k0)
    ms = _time_sorts(steps, warmup, lambda: (k.copy_(k0), v.copy_(v0)), lambda: s.sort_pairs(k, v), stream)
    prof = s.last_profile()
    pass_ms = float(np.mean(prof[2:]))
    ok = s.validate(k) == 0 and multiset_checksum(k) == ck
    # payload round trip on a slice: output key i is the input key at index v[i]
    idx = v[: 1 << 22].to(torch.int64) & 0xFFFFFFFF
    ok = ok and bool(torch.equal(k0[idx], k[: 1 << 22]))
    s.close()
    del k0, v0, k, v, idx
    torch.cuda.empty_cache()
    ach = 16 * n / (pass_ms / 1e3) / 1e9
    return {"workload": f"2^{n.bit_length() - 1} (uint32 key, uint32 payload) pairs, uniform-random keys, payload = index (BASELINE.json configs[2])",
            "value": round(n / (ms / 1e3) / 1e9, 3), "unit": "Gpairs/s", "ms_per_step": round(ms, 4), "steps": steps, "warmup": warmup,
            "passes": 4, "pct_of_peak_64B_per_pair": round(64.0 * n / (ms / 1e3) / 1e9 / peak * 100, 2),
            "roofline": {"bound": "hbm", "kernel": "digit_binning_wide_kernel<u32, pairs>", "achieved": round(ach, 1), "peak": peak,
                         "unit": "GB/s", "frac": round(ach / peak, 4), "algorithmic_bytes_per_launch": 16 * n, "launch_ms": round(pass_ms, 4)},
            "kernel_ms": {"global_histogram": round(prof[0], 4), "digit_binning_pass_mean": round(pass_ms, 4)}, "verified": bool(ok)}


def extra_config_u64(g, n, peak, steps=5, warmup=3):
    """BASELINE.json configs[3]: 2^30 uint64 keys-only (8 digit passes), device-timed, with its own roofline."""
    import numpy as np
    import torch

    w0 = torch.empty(2 * n, dtype=torch.int32, device="cuda")
    g.init_random(w0, 0, SEED)  # hi/lo words are consecutive draws of the reference generator
    k0 = w0.view(torch.int64)
    k = torch.empty_like(k0)
    s = g.OneSweepSorter(n, 8, 0)
    s.set_option("profile", 1)
    stream = torch.cuda.current_stream()
    ck = multiset_checksum(k0)
    ms = _time_sorts(steps, warmup, lambda: k.copy_(k0), lambda: s.sort_keys(k), stream)
    prof = s.last_profile()
    pass_ms = float(np.mean(prof[2:]))
    ok = s.validate(k) == 0 and multiset_checksum(k) == ck
    s.close()
    del w0, k0, k
    torch.cuda.empty_cache()
    ach = 16 * n / (pass_ms / 1e3) / 1e9
    return {"workload": f"2^{n.bit_length() - 1} uint64 keys-only, uniform-random, 8 digit passes (BASELINE.json configs[3])",
            "value": round(n / (ms / 1e3) / 1e9, 3), "unit": "Gkeys/s", "ms_per_step": round(ms, 4), "steps": steps, "warmup": warmup,
            "passes": 8, "pct_of_peak_128B_per_key": round(128.0 * n / (ms / 1e3) / 1e9 / peak * 100, 2),
            "roofline": {"bound": "hbm", "kernel": "digit_binning_wide_kernel<u64>", "achieved": round(ach, 1), "peak": peak,
                         "unit": "GB/s", "frac": round(ach / peak, 4), "algorithmic_bytes_per_launch": 16 * n, "launch_ms": round(pass_ms, 4)},
            "kernel_ms": {"global_histogram": round(prof[0], 4), "digit_binning_pass_mean": round(pass_ms, 4)}, "verified": bool(ok)}


def entropy_sweep(g, n, steps=3, warmup=2):
    """The reference's entropy benchmark (Thearling-Smith presets, UtilityKernels.cuh:42-52,70-81; chart README.md:27,
    protocol GPUSortingD3D12/Tests.h:383-393): and_count 0..4 ANDs 1..5 uniform draws (32 -> ~1 bit of entropy per key
    bit... 1.0, 0.811, 0.544, 0.337, 0.201 bits per bit), plus the degenerate cases that exercise pass skipping."""
    import torch

    src = torch.empty(n, dtype=torch.int32, device="cuda")
    work = torch.empty_like(src)
    s = g.OneSweepSorter(n, 4, 0)
    stream = torch.cuda.current_stream()
    out = []
    cases = [(f"entropy_preset_{a + 1}", a, None) for a in range(5)] + [("low_16_bits_only", 0, 0xFFFF), ("all_equal", 0, 0)]
    for name, andc, mask in cases:
        g.init_random(src, andc, SEED)
        if mask is not None:
            src &= mask
        ms = _time_sorts(steps, warmup, lambda: work.copy_(src), lambda: s.sort_keys(work), stream)
        ok = s.validate(work) == 0
        out.append({"input": name, "value": round(n / (ms / 1e3) / 1e9, 2), "unit": "Gkeys/s", "ms_per_sort": round(ms, 4),
                    "executed_passes": s.info("last_executed_passes"), "sorted": bool(ok)})
    s.close()
    del src, work
    torch.cuda.empty_cache()
    return out


def ref_cuda_leg(n):
    """The reference's own CUDA OneSweep kernels (oracle/_ref, compiled for sm_100a from /root/reference) timed in this
    process on this GPU with the reference's protocol (OneSweepDispatcher.cuh:193-239: InitRandom(seed+i) per iteration,
    cudaEvent around the dispatch incl. its memsets, iteration 0 discarded).  A measured comparator only."""
    import torch
    from tests import oraclelib

    ref = oraclelib.load_ref()
    if ref is None:
        return {"unavailable": "oracle/_ref/libref_onesweep.so not built"}
    out = {"what": "b0nes164/GPUSorting GPUSortingCUDA OneSweep kernels, unmodified but for the SURVEY D4 pragma token, sm_100a build, "
                   "timed with the reference's BatchTimingKeysOnly protocol", "unit": "Gkeys/s"}
    for e, iters in ((28, 20), (n.bit_length() - 1, 5)):
        m = 1 << e
        h = ref.lib.ref_create(m)
        a, alt = torch.empty(m, dtype=torch.int32, device="cuda"), torch.empty(m, dtype=torch.int32, device="cuda")
        total_ms = float(ref.lib.ref_batch_timing_keys(h, a.data_ptr(), alt.data_ptr(), m, iters, SEED))
        bad = int(ref.lib.ref_validate_keys(h, a.data_ptr(), m))
        ref.lib.ref_destroy(h)
        del a, alt
        torch.cuda.empty_cache()
        out[f"keys_2pow{e}"] = {"value": round(m * iters / (total_ms / 1e3) / 1e9, 3), "ms_per_sort": round(total_ms / iters, 4),
                                "iters": iters, "sorted": bad == 0}
    return out


def bench_single(args, g, n, device_index):
    import numpy as np
    import torch

    src = torch.empty(n, dtype=torch.int32, device="cuda")
    g.init_random(src, 0, SEED)
    work = torch.empty_like(src)
    s = g.OneSweepSorter(n, 4, 0)
    variant = int(os.environ.get("OSB_VARIANT", s.info("variant")))
    s.set_option("variant", variant)
    s.set_option("profile", 1)
    stream = torch.cuda.current_stream()
    checksum_in = multiset_checksum(src)

    def one_step(timed):
        work.copy_(src)  # restore the unsorted input (untimed)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        s.sort_keys(work)
        b.record(stream)
        return (a, b)

    for _ in range(args.warmup):
        one_step(False)
    torch.cuda.synchronize()
    # the handle's pass counter advances once per digit place of every multi-kernel sort (4 for uint32 keys), so it counts
    # the sorts the timed loop really issued (bench sizes are far above the one-launch small-n path, which has no pass)
    epoch0 = s.info("epoch")
    sampler = ClockSampler(device_index)
    sampler.start()
    events, profiles = [], []
    torch.cuda.synchronize()
    for _ in range(args.steps):
        events.append(one_step(True))
        profiles.append(s.last_profile())  # waits for this sort's last event only
    torch.cuda.synchronize()
    clocks = sampler.result()
    ms = sum(a.elapsed_time(b) for a, b in events) / args.steps
    prof = np.array(profiles)  # [steps][hist, scan, pass0..3]
    kernel_ms = {"global_histogram": float(prof[:, 0].mean()), "scan": float(prof[:, 1].mean()),
                 "digit_binning_pass_mean": float(prof[:, 2:].mean())}
    for p in range(prof.shape[1] - 2):
        kernel_ms[f"digit_binning_pass_{p}"] = float(prof[:, 2 + p].mean())
    timed_sorts = (s.info("epoch") - epoch0) // 4
    # sorted (the reference's Validate) AND the same multiset as the input (an output of equal keys would not pass)
    verified = s.validate(work) == 0 and multiset_checksum(work) == checksum_in
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"sorted_keys": work})
    launches = s.info("launches_per_sort")

    # ---- end to end through the C-ABI host entry point, pinned host memory ---------------------------------
    e2e_steps = max(1, min(args.e2e_steps, args.steps))
    host_src = torch.empty(n, dtype=torch.int32).pin_memory()
    host_src.copy_(src)
    host_work = torch.empty(n, dtype=torch.int32).pin_memory()
    del src, work
    torch.cuda.empty_cache()
    total = 0.0
    for i in range(e2e_steps + 1):
        host_work.copy_(host_src)  # untimed restore
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        s.sort_host(host_work)  # H2D + sort + D2H + sync inside
        dt = time.perf_counter() - t0
        if i:
            total += dt
    e2e_ms = total / e2e_steps * 1e3
    hw = host_work.numpy().view(np.uint32)
    verified = verified and bool((hw[:-1][:: 4097] <= hw[1:][:: 4097]).all())
    verified = verified and int(hw.sum(dtype=np.uint64)) == checksum_in[0]
    tile_keys, rank_mode = s.info("tile_keys"), s.info("rank_mode")
    s.close()
    del host_src, host_work, hw
    torch.cuda.empty_cache()
    out = {
        "ms_per_step": ms, "pass_ms": kernel_ms["digit_binning_pass_mean"], "kernel_ms": kernel_ms,
        "kernel": "digit_binning_wide_kernel" if variant == 2 else ("digit_binning_persistent_kernel" if variant == 1 else "digit_binning_tile_kernel"),
        "variant": variant, "tile_keys": tile_keys, "rank_mode": "atomic" if rank_mode == 0 else "ballot",
        "e2e_ms_per_step": e2e_ms, "e2e_steps": e2e_steps, "h2d_bytes": 4 * n, "d2h_bytes": 4 * n,
        "gpu_launches": timed_sorts * launches, "clocks": clocks, "verified": verified,
    }
    if not args.no_extra:
        peak, _ = measured_peak_gbs()
        out["extra_configs"] = [extra_config_pairs(g, n, peak), extra_config_u64(g, n, peak)]
        out["ref_cuda"] = ref_cuda_leg(n)
        out["entropy_sweep"] = entropy_sweep(g, n)
    return out


if __name__ == "__main__":
    main()
