"""ctypes access to the TEST-ONLY libraries under oracle/ (the CPU restatement and, when built, the
reference's own CUDA kernels), and the tensor digest the golden fixtures store.  Only tests/, __graft_entry__.smoke()
and bench.py's CPU-baseline legs may import this module; nothing under gpusorting_b200/ does."""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_SO = os.path.join(ROOT, "oracle", "build", "liboracle.so")
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libref_onesweep.so")

u64, u32, vp, ci = ctypes.c_uint64, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_int


class Oracle:
    def __init__(self, lib):
        self.lib = lib
        sig = {
            "orc_init_random_u32": (None, [vp, u64, u32, u32]),
            "orc_init_random_pairs_u32": (None, [vp, vp, u64, u32, u32]),
            "orc_init_random_u64": (None, [vp, u64, u32, u32]),
            "orc_global_histogram": (None, [vp, u64, ci, vp]),
            "orc_scan_exclusive": (None, [vp, ci, vp]),
            "orc_binning_pass_u32": (None, [vp, vp, vp, vp, u64, u32]),
            "orc_binning_pass_u64": (None, [vp, vp, u64, u32]),
            "orc_onesweep_keys_u32": (ci, [vp, vp, u64]),
            "orc_onesweep_pairs_u32": (ci, [vp, vp, vp, vp, u64]),
            "orc_onesweep_keys_u64": (ci, [vp, vp, u64]),
            "orc_validate_keys_u32": (u64, [vp, u64]),
            "orc_validate_keys_u64": (u64, [vp, u64]),
            "orc_validate_pairs_u32": (u64, [vp, vp, u64]),
            "orc_onesweep_parallel": (ci, [vp, vp, vp, vp, u64, ci, ci]),
            "orc_host_threads": (ci, []),
            "orc_digest": (u64, [vp, u64]),
            "orc_std_sort_u32": (None, [vp, u64]),
            "orc_std_sort_u64": (None, [vp, u64]),
            "orc_parallel_sort_u32": (None, [vp, u64, ci]),
            "orc_parallel_sort_u64": (None, [vp, u64, ci]),
            "orc_std_stable_sort_pairs_u32": (None, [vp, vp, u64]),
        }
        for name, (res, args) in sig.items():
            f = getattr(lib, name)
            f.restype, f.argtypes = res, args

    # ---- inputs ------------------------------------------------------------------------------------
    def init_random_u32(self, n, and_count=0, seed=10):
        k = np.empty(n, np.uint32)
        self.lib.orc_init_random_u32(k.ctypes.data, n, and_count, seed)
        return k

    def init_random_u64(self, n, and_count=0, seed=10):
        k = np.empty(n, np.uint64)
        self.lib.orc_init_random_u64(k.ctypes.data, n, and_count, seed)
        return k

    # ---- the algorithm -----------------------------------------------------------------------------
    def global_histogram(self, keys):
        kb = keys.dtype.itemsize
        h = np.zeros(kb * 256, np.uint64)
        self.lib.orc_global_histogram(keys.ctypes.data, keys.size, kb, h.ctypes.data)
        return h.reshape(kb, 256)

    def scan_exclusive(self, hist):
        h = np.ascontiguousarray(hist, np.uint64)
        out = np.empty_like(h)
        self.lib.orc_scan_exclusive(h.ctypes.data, h.shape[0], out.ctypes.data)
        return out

    def binning_pass(self, keys, shift, vals=None):
        dst = np.empty_like(keys)
        if keys.dtype == np.uint64:
            self.lib.orc_binning_pass_u64(keys.ctypes.data, dst.ctypes.data, keys.size, shift)
            return dst
        if vals is None:
            self.lib.orc_binning_pass_u32(keys.ctypes.data, dst.ctypes.data, None, None, keys.size, shift)
            return dst
        dv = np.empty_like(vals)
        self.lib.orc_binning_pass_u32(keys.ctypes.data, dst.ctypes.data, vals.ctypes.data, dv.ctypes.data, keys.size, shift)
        return dst, dv

    def sort_keys(self, keys):
        k = keys.copy()
        alt = np.empty_like(k)
        fn = self.lib.orc_onesweep_keys_u32 if k.dtype == np.uint32 else self.lib.orc_onesweep_keys_u64
        fn(k.ctypes.data, alt.ctypes.data, k.size)
        return k

    def sort_pairs(self, keys, vals):
        k, v = keys.copy(), vals.copy()
        ak, av = np.empty_like(k), np.empty_like(v)
        self.lib.orc_onesweep_pairs_u32(k.ctypes.data, v.ctypes.data, ak.ctypes.data, av.ctypes.data, k.size)
        return k, v

    def sort_parallel_inplace(self, keys, vals=None, threads=0, alt=None):
        alt = np.empty_like(keys) if alt is None else alt
        av = np.empty_like(vals) if vals is not None else None
        return self.lib.orc_onesweep_parallel(keys.ctypes.data, alt.ctypes.data,
                                              vals.ctypes.data if vals is not None else None,
                                              av.ctypes.data if av is not None else None,
                                              keys.size, keys.dtype.itemsize, threads)

    def validate(self, keys):
        fn = self.lib.orc_validate_keys_u32 if keys.dtype == np.uint32 else self.lib.orc_validate_keys_u64
        return int(fn(keys.ctypes.data, keys.size))

    def digest(self, arr):
        a = np.ascontiguousarray(arr)
        return int(self.lib.orc_digest(a.ctypes.data, a.nbytes))

    def host_threads(self):
        return int(self.lib.orc_host_threads())


def build_oracle():
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "oracle"], check=True)


def load_oracle() -> Oracle:
    if not os.path.exists(ORACLE_SO):
        build_oracle()
    return Oracle(ctypes.CDLL(ORACLE_SO))


def device_digest(t) -> int:
    """Order-sensitive 64-bit checksum of a tensor's 32-bit words, computed where the tensor lives.  Each word is mixed with
    its index and the mixes are summed with wrapping int64 arithmetic, so the value does not depend on reduction order;
    moving a word to another index changes it.  Digests of the reference's 2^30-element outputs are stored under
    tests/golden/, where a host-side hash of 4 GiB per array would take seconds each."""
    import torch

    flat = t.reshape(-1).view(torch.int32)
    k1, k2 = 0x2545F4914F6CDD1D, 0x5851F42D4C957F2D
    h, step = 0, 1 << 26
    for s in range(0, flat.numel(), step):
        x = flat[s:s + step].to(torch.int64) & 0xFFFFFFFF
        i = torch.arange(s, s + x.numel(), dtype=torch.int64, device=x.device)
        y = (x ^ (i * k1)) * k2
        y = (y ^ (y >> 29)) * k1
        h += int(y.sum().item())
    return h & ((1 << 64) - 1)


class RefCuda:
    """The reference's own kernels behind oracle/ref_harness.cu (needs a GPU)."""

    def __init__(self, lib):
        self.lib = lib
        f32 = ctypes.c_float
        sig = {
            "ref_create": (vp, [u32]),
            "ref_destroy": (None, [vp]),
            "ref_init_random_keys": (ci, [vp, u32, u32, u32]),
            "ref_init_random_pairs": (ci, [vp, vp, u32, u32, u32]),
            "ref_sort_keys": (ci, [vp, vp, vp, u32]),
            "ref_sort_pairs": (ci, [vp, vp, vp, vp, vp, u32]),
            "ref_get_global_histogram": (ci, [vp, vp]),
            "ref_validate_keys": (ctypes.c_longlong, [vp, vp, u32]),
            "ref_validate_pairs": (ctypes.c_longlong, [vp, vp, vp, u32]),
            "ref_batch_timing_keys": (f32, [vp, vp, vp, u32, u32, u32]),
            "ref_batch_timing_pairs": (f32, [vp, vp, vp, vp, vp, u32, u32, u32]),
        }
        for name, (res, args) in sig.items():
            f = getattr(lib, name)
            f.restype, f.argtypes = res, args


def load_ref():
    if not os.path.exists(REF_SO):
        return None
    try:
        return RefCuda(ctypes.CDLL(REF_SO))
    except OSError:
        return None
