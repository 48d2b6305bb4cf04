"""Multi-GPU sharded OneSweep: one process per GPU, MSD bucket exchange over NVLink, then a local OneSweep.

No reference equivalent (the reference is single-device, SURVEY 2.1) -- this is BASELINE.json's fifth config.
torch.distributed is the plumbing only (rendezvous, broadcasting the NCCL unique id, reducing timings); the
exchange itself runs inside libonesweep_b200.so (osb_sharded.cu): by default the DigitBinningPass kernel scatters
straight into the peers' CUDA-IPC-mapped receive buffers over NVLink ("fused"), with ncclSend/ncclRecv of a locally
partitioned buffer as the staged baseline.
"""
from __future__ import annotations

import ctypes
import time
from typing import Optional

import numpy as np
import torch
import torch.distributed as dist

from ._lib import check, lib


def plan(hist_all: np.ndarray, rank: int):
    """Host-side exchange plan (pure function; usable without a GPU): see osb200_sharded_plan in the header.

    hist_all: [world, 256] uint64 most-significant-digit counts of every rank.
    Returns (dest[256] int32, recv_count[world] uint64, recv_off[256] uint64 for source `rank`)."""
    h = np.ascontiguousarray(hist_all, dtype=np.uint64)
    world = h.shape[0]
    dest = np.empty(256, np.int32)
    recv_count = np.empty(world, np.uint64)
    recv_off = np.empty(256, np.uint64)
    check(lib.osb200_sharded_plan(h.ctypes.data, world, int(rank), dest.ctypes.data, recv_count.ctypes.data,
                                  recv_off.ctypes.data), "osb200_sharded_plan")
    return dest, recv_count, recv_off


class _DevicePtr:
    """Zero-copy view of handle-owned device memory as a torch tensor (CUDA array interface)."""

    def __init__(self, ptr: int, n: int, typestr: str = "<i4"):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 3}


class ShardedSorter:
    def __init__(self, max_n_local: int, slack_percent: int = 25, group=None):
        if not dist.is_initialized():
            raise RuntimeError("torch.distributed must be initialised (one process per GPU)")
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        uid = torch.zeros(128, dtype=torch.uint8)
        if self.rank == 0:
            buf = (ctypes.c_uint8 * 128)()
            check(lib.osb200_sharded_unique_id(buf), "osb200_sharded_unique_id")
            uid = torch.tensor(list(buf), dtype=torch.uint8)
        backend = dist.get_backend(group)
        if backend == "nccl":
            uid = uid.cuda()
        dist.broadcast(uid, src=0, group=group)
        raw = bytes(uid.cpu().tolist())
        h = ctypes.c_void_p()
        check(lib.osb200_sharded_create(ctypes.byref(h), raw, self.rank, self.world, int(max_n_local), int(slack_percent)),
              "osb200_sharded_create")
        self._h = h
        self.max_n_local = int(max_n_local)
        self._stage = None
        self._host_out = None

    def close(self):
        if getattr(self, "_h", None):
            lib.osb200_sharded_destroy(self._h)
            self._h = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def set_fused(self, fused: bool) -> None:
        check(lib.osb200_sharded_set_fused(self._h, 1 if fused else 0), "osb200_sharded_set_fused")

    def force_fine(self, on: bool) -> None:
        check(lib.osb200_sharded_force_fine(self._h, 1 if on else 0), "osb200_sharded_force_fine")

    def set_local_option(self, key: str, value: int) -> None:
        a, b = ctypes.c_void_p(), ctypes.c_void_p()
        check(lib.osb200_sharded_local_handle(self._h, ctypes.byref(a), ctypes.byref(b)), "osb200_sharded_local_handle")
        for hh in (a, b):
            check(lib.osb200_set_option(hh, key.encode(), int(value)), f"osb200_set_option({key})")

    def local_profile(self):
        """Per-kernel ms of the last LOCAL OneSweep on this rank ([hist, scan, pass0..3]) when option 'profile' was set
        through set_local_option: the local handle's own CUDA events, not an estimate."""
        a, b = ctypes.c_void_p(), ctypes.c_void_p()
        check(lib.osb200_sharded_local_handle(self._h, ctypes.byref(a), ctypes.byref(b)), "osb200_sharded_local_handle")
        buf = (ctypes.c_float * 16)()
        k = lib.osb200_get_profile(b, buf, 16)
        if k < 0:
            check(k, "osb200_get_profile")
        return [float(buf[i]) for i in range(k)]

    def local_info(self, key: str) -> int:
        a, b = ctypes.c_void_p(), ctypes.c_void_p()
        check(lib.osb200_sharded_local_handle(self._h, ctypes.byref(a), ctypes.byref(b)), "osb200_sharded_local_handle")
        return int(lib.osb200_get_info(b, key.encode()))

    def sort_keys(self, keys: torch.Tensor, n_local: Optional[int] = None, stream=None) -> torch.Tensor:
        """keys: this rank's unsorted int32/uint32 CUDA tensor (not modified).  Returns this rank's slice of the global
        ascending order as a tensor that aliases sorter-owned memory (valid until the next call)."""
        n_local = keys.numel() if n_local is None else int(n_local)
        if not (isinstance(keys, torch.Tensor) and keys.is_cuda and keys.is_contiguous() and keys.dim() == 1
                and keys.dtype in (torch.int32, torch.uint32)):
            raise TypeError("keys must be a contiguous 1-D int32/uint32 CUDA tensor")
        if keys.device.index != torch.cuda.current_device():
            raise ValueError("keys must live on this rank's current CUDA device")
        if not (0 <= n_local <= keys.numel()):
            raise ValueError(f"n_local={n_local} is outside 0..keys.numel()={keys.numel()}")
        s = stream if stream is not None else torch.cuda.current_stream()
        out, n_out = ctypes.c_void_p(), ctypes.c_uint64(0)
        check(lib.osb200_sharded_sort_keys_u32(self._h, keys.data_ptr(), n_local, ctypes.byref(out), ctypes.byref(n_out),
                                               int(s.cuda_stream)), "osb200_sharded_sort_keys_u32")
        if n_out.value == 0:
            return torch.empty(0, dtype=torch.int32, device=keys.device)
        return torch.as_tensor(_DevicePtr(out.value, int(n_out.value)), device=keys.device)

    def sort_host(self, host_keys: torch.Tensor) -> torch.Tensor:
        """End to end: pinned (or pageable) host keys in, this rank's sorted slice back on the host."""
        n = host_keys.numel()
        if self._stage is None or self._stage.numel() < n:
            self._stage = torch.empty(self.max_n_local, dtype=torch.int32, device="cuda")
        self._stage[:n].copy_(host_keys, non_blocking=True)
        res = self.sort_keys(self._stage, n)
        if self._host_out is None or self._host_out.numel() < res.numel():  # pinned once, reused by later calls
            cap = max(res.numel(), self.max_n_local + self.max_n_local // 4)
            self._host_out = torch.empty(cap, dtype=torch.int32, pin_memory=True)
        out = self._host_out[: res.numel()]
        out.copy_(res, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return out

    def last_timing(self):
        buf = (ctypes.c_float * 4)()
        check(lib.osb200_sharded_last_timing(self._h, buf), "osb200_sharded_last_timing")
        return {"histogram_allgather_plan_ms": buf[0], "exchange_ms": buf[1], "local_sort_ms": buf[2], "total_ms": buf[3]}


def verify_global_order(res: torch.Tensor, rank: int, world: int) -> bool:
    """Every rank's slice is sorted and slices are ordered across ranks (boundary check via all_gather)."""
    from .onesweep import OneSweepSorter

    ok = True
    if res.numel() > 1:
        ok = bool((res[1:].to(torch.int64) & 0xFFFFFFFF >= res[:-1].to(torch.int64) & 0xFFFFFFFF).all())
    lo = int(res[0].item()) & 0xFFFFFFFF if res.numel() else -1
    hi = int(res[-1].item()) & 0xFFFFFFFF if res.numel() else -1
    t = torch.tensor([lo, hi, res.numel()], dtype=torch.int64, device="cuda")
    allb = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(allb, t)
    prev_hi = -1
    for b in allb:
        blo, bhi, cnt = (int(x) for x in b)
        if cnt == 0:
            continue
        ok = ok and blo >= prev_hi
        prev_hi = bhi
    return ok


def global_multiset_checksum(t: torch.Tensor) -> tuple:
    """Order-independent checksum (sum and a mixed sum of the 32-bit words, mod 2^63) all-reduced over the ranks: equal
    before and after a sharded sort iff no key was lost, duplicated or replaced (up to hash collisions)."""
    a = torch.zeros(2, dtype=torch.int64, device="cuda")
    flat = t.view(torch.int32)
    step = 1 << 27
    for i in range(0, flat.numel(), step):
        x = flat[i:i + step].to(torch.int64) & 0xFFFFFFFF
        a[0] += x.sum()
        a[1] += ((x * 2654435761) ^ (x >> 7)).sum()
    dist.all_reduce(a)  # int64 wrap-around is still a function of the multiset only
    return int(a[0]), int(a[1])


def bench_sharded(args, rank: int, world: int, local_rank: int, n: int):
    """bench.py body for N>1: weak scaling, 2^30 keys per rank (seed 10+rank), sharded sort timed on the device."""
    import os

    from . import init_random
    from .onesweep import OneSweepSorter  # noqa: F401

    from bench import DUMP_SAMPLE, SEED, ClockSampler, dump_outputs  # type: ignore

    src = torch.empty(n, dtype=torch.int32, device="cuda")
    init_random(src, 0, SEED + rank)
    s = ShardedSorter(n, slack_percent=int(os.environ.get("OSB_SLACK", "12")))
    if os.environ.get("OSB_FUSED") is not None:
        s.set_fused(os.environ["OSB_FUSED"] != "0")
    s.set_local_option("profile", 1)
    total_in = torch.tensor([n], dtype=torch.int64, device="cuda")
    dist.all_reduce(total_in)
    checksum_in = global_multiset_checksum(src)
    stream = torch.cuda.current_stream()

    def one_step():
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        res = s.sort_keys(src)
        b.record(stream)
        return a, b, res

    for _ in range(args.warmup):
        one_step()
    torch.cuda.synchronize()
    dist.barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    torch.cuda.synchronize()
    # The host does not wait for the GPU between the steps (each step still has its one host wait inside the call, for the
    # plan): it enqueues step i+1's histogram while step i's local sort runs, as a pipelining caller would.  Waiting here after
    # every step put every host stall (10-20 ms ones were seen with >= 4 ranks on a box) on the critical path of ALL ranks
    # through the next collective.  The phase times reported are those of the last timed step.
    events, phases, local_prof = [], [], []
    for _ in range(args.steps):
        a, b, res = one_step()
        events.append((a, b))
    torch.cuda.synchronize()
    phases.append(s.last_timing())
    local_prof.append(s.local_profile())
    dist.barrier()
    clocks = sampler.result()
    ms = sum(a.elapsed_time(b) for a, b in events) / args.steps
    total_out = torch.tensor([res.numel()], dtype=torch.int64, device="cuda")
    dist.all_reduce(total_out)
    verified = (verify_global_order(res, rank, world) and int(total_out) == int(total_in)
                and global_multiset_checksum(res) == checksum_in)
    if args.dump_outputs:  # this rank's slice of the global order, as ShardedSorter.sort_keys returned it
        dump_outputs(args.dump_outputs, {f"sorted_keys_rank{rank}": res}, DUMP_SAMPLE // world)
    ph = {k: float(np.mean([p[k] for p in phases])) for k in phases[0]}
    # every rank's own view (phases are measured by the rank's own CUDA events; a rank that arrives early at a collective
    # waits inside the phase that contains it)
    mine = torch.tensor([ms] + [ph[k] for k in sorted(ph)], dtype=torch.float64, device="cuda")
    allv = [torch.zeros_like(mine) for _ in range(world)]
    dist.all_gather(allv, mine)
    per_rank = [dict(zip(["ms_per_step"] + sorted(ph), (round(float(x), 4) for x in v))) for v in allv]

    # end to end: pinned host keys in, sorted slice back out
    e2e_steps = max(1, min(args.e2e_steps, args.steps))
    host = torch.empty(n, dtype=torch.int32).pin_memory()
    host.copy_(src)
    tot = 0.0
    for i in range(e2e_steps + 1):
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        out = s.sort_host(host)
        dt = time.perf_counter() - t0
        if i:
            tot += dt
    e2e_ms = tot / e2e_steps * 1e3
    # the local sort's DigitBinningPass time: this rank's local handle recorded CUDA events between its kernels
    lp = np.array(local_prof)  # [steps][hist, scan, pass0..]
    local_pass_ms = float(lp[:, 2:].mean())
    ph["local_global_histogram_ms"] = float(lp[:, 0].mean())
    ph["local_digit_binning_pass_mean_ms"] = local_pass_ms
    # kernels launched per sharded sort: MSD histogram + exchange pass (+ its scan in staged mode) + the local sort's
    launches_per_sort = 1 + 1 + s.local_info("launches_per_sort")
    result = {
        "ms_per_step": ms, "pass_ms": local_pass_ms, "kernel_ms": ph, "phases_ms": ph, "per_rank": per_rank,
        "kernel": "digit_binning_wide_kernel (local sort) + fused NVLink exchange pass",
        "variant": s.local_info("variant"), "tile_keys": s.local_info("tile_keys"),
        "rank_mode": "atomic" if s.local_info("rank_mode") == 0 else "ballot", "e2e_ms_per_step": e2e_ms, "e2e_steps": e2e_steps,
        "h2d_bytes": 4 * n, "d2h_bytes": 4 * int(out.numel()), "gpu_launches": args.steps * launches_per_sort, "clocks": clocks,
        "verified": bool(verified),
        "e2e_api": "ShardedSorter.sort_host: torch pinned H2D copy + osb200_sharded_sort_keys_u32 (C-ABI) + torch D2H copy of the slice",
    }
    s.close()
    return result
