"""Generate the golden fixtures under tests/golden/ from THE REFERENCE ITSELF.

Run on a B200 after `make -C oracle ref` has built oracle/_ref/libref_onesweep.so (the reference's own
OneSweep.cu / UtilityKernels.cuh behind oracle/ref_harness.cu):
    python tests/golden/make_ref_golden.py OUT_DIR
then copy OUT_DIR/*.json into tests/golden/.  No product code is involved.

ref_onesweep_golden.json: InitRandom<<<256,256>>> (UtilityKernels.cuh:53-117) then the dispatcher's launch order
(OneSweepDispatcher.cuh:311-363), with small order-sensitive host digests (FNV-1a 64) plus the first/last elements,
for sizes the CPU oracle re-computes in seconds.

ref_onesweep_parity_golden.json: device digests (oraclelib.device_digest) of the reference's inputs and outputs for the
GPU parity tests -- test_gpu_parity.test_bit_exact_vs_reference_cuda and the 2^30 cases of test_gpu_fullsize -- so that
they compare with the reference on a machine where oracle/_ref cannot be built.
"""
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from tests import oraclelib  # noqa: E402
from tests.oraclelib import device_digest  # noqa: E402

CASES = [  # (n, and_count, seed, pairs)
    (7680, 0, 7680, False),      # the first size of the reference's TestAllKeysOnly sweep (seed == n)
    (7681, 0, 7681, False),
    (12345, 0, 12345, True),
    (15360, 0, 15360, False),
    (65537, 0, 10, False),       # wraps the 65,536-stream generator
    (1 << 20, 0, 10, False),     # BASELINE.json configs[0]
    (1 << 20, 0, 10, True),
    (1 << 20, 1, 10, False),     # entropy presets 2..5 (Thearling-Smith AND-ing)
    (1 << 20, 2, 10, False),
    (1 << 20, 3, 10, False),
    (1 << 20, 4, 10, False),
    (1 << 22, 0, 22, False),
]

BIT_EXACT_SIZES = [(7680, 7680), (9999, 9999), (1 << 20, 10), (1 << 22, 22)]  # (n, seed), keys and pairs each
FULL_N = 1 << 30  # the reference is valid up to exactly 2^30 (30-bit descriptor value, SURVEY D5)


def make_golden(ref, orc):
    max_n = max(c[0] for c in CASES)
    h = ref.lib.ref_create(max_n)
    assert h
    sort = torch.empty(max_n, dtype=torch.int32, device="cuda")
    alt = torch.empty_like(sort)
    pay = torch.empty_like(sort)
    altpay = torch.empty_like(sort)
    out = {"generator": "tests/golden/make_ref_golden.py", "source": "reference CUDA kernels via oracle/_ref", "cases": []}
    for n, andc, seed, pairs in CASES:
        if pairs:
            assert ref.lib.ref_init_random_pairs(sort.data_ptr(), pay.data_ptr(), n, andc, seed) == 0
        else:
            assert ref.lib.ref_init_random_keys(sort.data_ptr(), n, andc, seed) == 0
        torch.cuda.synchronize()
        inp = sort[:n].cpu().numpy().view(np.uint32).copy()
        if pairs:
            assert ref.lib.ref_sort_pairs(h, sort.data_ptr(), pay.data_ptr(), alt.data_ptr(), altpay.data_ptr(), n) == 0
        else:
            assert ref.lib.ref_sort_keys(h, sort.data_ptr(), alt.data_ptr(), n) == 0
        torch.cuda.synchronize()
        res = sort[:n].cpu().numpy().view(np.uint32).copy()
        hist = np.empty(1024, np.uint32)
        assert ref.lib.ref_get_global_histogram(h, hist.ctypes.data) == 0
        errs = int(ref.lib.ref_validate_keys(h, sort.data_ptr(), n))
        case = {
            "n": n, "and_count": andc, "seed": seed, "pairs": pairs,
            "input_head": [int(x) for x in inp[:8]], "input_digest": orc.digest(inp),
            "sorted_head": [int(x) for x in res[:8]], "sorted_tail": [int(x) for x in res[-8:]],
            "sorted_digest": orc.digest(res), "global_hist_digest": orc.digest(hist.astype(np.uint64)),
            "ref_validate_errors": errs,
        }
        if pairs:
            pres = pay[:n].cpu().numpy().view(np.uint32).copy()
            case["payload_digest"] = orc.digest(pres)
        out["cases"].append(case)
        print(n, andc, seed, pairs, "ok", hex(case["sorted_digest"]))
    ref.lib.ref_destroy(h)
    return out


def _sorted_case(ref, k, v, n):
    """Digests of the input in k (and v), the reference's sort of it and its validator's verdict; k, v sorted in place."""
    h = ref.lib.ref_create(n)
    assert h
    case = {"input_digest": device_digest(k)}
    if v is not None:
        case["input_payload_digest"] = device_digest(v)
    ak = torch.empty_like(k)
    if v is None:
        assert ref.lib.ref_sort_keys(h, k.data_ptr(), ak.data_ptr(), n) == 0
    else:
        av = torch.empty_like(v)
        assert ref.lib.ref_sort_pairs(h, k.data_ptr(), v.data_ptr(), ak.data_ptr(), av.data_ptr(), n) == 0
        del av
    torch.cuda.synchronize()
    del ak
    case["sorted_digest"] = device_digest(k)
    if v is not None:
        case["payload_digest"] = device_digest(v)
    case["ref_validate_errors"] = int(ref.lib.ref_validate_keys(h, k.data_ptr(), n))
    assert case["ref_validate_errors"] == 0
    ref.lib.ref_destroy(h)
    torch.cuda.empty_cache()
    return case


def make_parity_golden(ref):
    out = {"generator": "tests/golden/make_ref_golden.py", "source": "reference CUDA kernels via oracle/_ref",
           "digest": "tests/oraclelib.py device_digest", "bit_exact": [], "fullsize": {}}
    for n, seed in BIT_EXACT_SIZES:
        k = torch.empty(n, dtype=torch.int32, device="cuda")
        v = torch.empty_like(k)
        assert ref.lib.ref_init_random_keys(k.data_ptr(), n, 0, seed) == 0
        keys = _sorted_case(ref, k, None, n)
        assert ref.lib.ref_init_random_pairs(k.data_ptr(), v.data_ptr(), n, 0, seed) == 0  # payload = key
        pairs = _sorted_case(ref, k, v, n)
        out["bit_exact"].append({"n": n, "seed": seed, "keys": keys, "pairs": pairs})
        print("bit_exact", n, seed, "ok")
        del k, v
    n = FULL_N
    k = torch.empty(n, dtype=torch.int32, device="cuda")
    assert ref.lib.ref_init_random_keys(k.data_ptr(), n, 0, 10) == 0
    out["fullsize"]["keys_u32"] = dict(n=n, seed=10, **_sorted_case(ref, k, None, n))
    print("fullsize keys_u32 ok")
    # 20-bit keys (~1024 duplicates of every value), payload = index: the input of the stability comparison
    assert ref.lib.ref_init_random_keys(k.data_ptr(), n, 0, 10) == 0
    k &= 0xFFFFF
    v = torch.arange(n, dtype=torch.int32, device="cuda")
    out["fullsize"]["pairs_u32_index_payload"] = dict(n=n, seed=10, key_mask=0xFFFFF, **_sorted_case(ref, k, v, n))
    print("fullsize pairs_u32_index_payload ok")
    assert ref.lib.ref_init_random_pairs(k.data_ptr(), v.data_ptr(), n, 0, 10) == 0  # payload = key
    out["fullsize"]["pairs_u32_key_payload"] = dict(n=n, seed=10, **_sorted_case(ref, k, v, n))
    print("fullsize pairs_u32_key_payload ok")
    return out


def main(out_dir):
    ref = oraclelib.load_ref()
    orc = oraclelib.load_oracle()
    assert ref is not None, "oracle/_ref/libref_onesweep.so missing"
    os.makedirs(out_dir, exist_ok=True)
    for name, data in (("ref_onesweep_golden.json", make_golden(ref, orc)),
                       ("ref_onesweep_parity_golden.json", make_parity_golden(ref))):
        with open(os.path.join(out_dir, name), "w") as f:
            json.dump(data, f, indent=1)


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: python tests/golden/make_ref_golden.py OUT_DIR  (writes OUT_DIR/ref_onesweep_golden.json and "
                 "OUT_DIR/ref_onesweep_parity_golden.json)")
    main(sys.argv[1])
