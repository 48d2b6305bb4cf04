"""BASELINE.json's full sizes (2^30) through size-independent properties: sortedness (the reference's Validate),
conservation of every digit-place histogram, a multiset checksum, stability via payload order, and bit-exact
equality with the reference's CUDA OneSweep through device digests of its outputs (tests/golden/).  Needs a B200: -m gpu."""
import json
import os

import numpy as np
import pytest
import torch

from tests.oraclelib import device_digest

pytestmark = pytest.mark.gpu

PARITY_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_onesweep_parity_golden.json")


def reference_case(name):
    """Digests of the input and of the reference CUDA OneSweep's output for one 2^30 case (tests/golden/make_ref_golden.py)."""
    return json.load(open(PARITY_GOLDEN))["fullsize"][name]


def multiset_checksum(t):
    """Order-independent: wrapping sums of x, x*x and x*2654435761 over all elements, in chunks to bound memory."""
    a = b = c = 0
    flat = t.view(torch.int32)
    step = 1 << 28
    for i in range(0, flat.numel(), step):
        x = flat[i:i + step].to(torch.int64) & 0xFFFFFFFF
        a += int(x.sum().item())
        b += int((x * x).sum().item())          # int64 arithmetic wraps: still a function of the multiset only
        c += int((x * 2654435761 ^ (x >> 7)).sum().item())
    m = (1 << 64) - 1
    return a & m, b & m, c & m


@pytest.fixture(scope="module")
def g():
    import gpusorting_b200 as g

    return g


def test_keys_u32_2pow30(g):
    n = 1 << 30
    ref = reference_case("keys_u32")  # the reference is valid up to exactly 2^30 (30-bit descriptor value, SURVEY D5)
    assert ref["n"] == n
    s = g.OneSweepSorter(n, 4, 0)
    t = torch.empty(n, dtype=torch.int32, device="cuda")
    g.init_random(t, 0, ref["seed"])
    assert device_digest(t) == ref["input_digest"]
    h0 = s.global_histogram(t).clone()
    c0 = multiset_checksum(t)
    s.sort_keys(t)
    assert s.validate(t) == 0
    assert torch.equal(s.global_histogram(t), h0)
    assert multiset_checksum(t) == c0
    assert device_digest(t) == ref["sorted_digest"], "keys differ from the reference CUDA OneSweep"
    # idempotence: sorting sorted data changes nothing
    first = t[: 1 << 20].clone()
    s.sort_keys(t)
    assert torch.equal(t[: 1 << 20], first) and s.validate(t) == 0
    s.close()


def test_pairs_u32_2pow30_stability(g):
    n = 1 << 30
    s = g.OneSweepSorter(n, 4, 4)
    k = torch.empty(n, dtype=torch.int32, device="cuda")
    v = torch.empty(n, dtype=torch.int32, device="cuda")
    g.init_random(k, 0, 10, payload=v, payload_is_index=True)
    k &= 0xFFFFF  # ~1024 duplicates per key value: stability is observable
    kin = k.clone()
    s.sort_pairs(k, v)
    assert s.validate(k) == 0
    # payload round trip: output key i must be the input key at index v[i]
    idx = v.view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    assert torch.equal(kin[idx], k)
    del kin, idx
    # stability: inside every run of equal keys the original indices ascend
    same = k[1:] == k[:-1]
    vi = v.to(torch.int64) & 0xFFFFFFFF
    assert bool(((vi[1:] > vi[:-1]) | ~same).all())
    s.close()


def test_pairs_u32_2pow30_bit_exact_vs_reference_cuda(g):
    """BASELINE config 3 as SURVEY 8(d) states it: 2^30 (key, payload) pairs, keys AND payloads bit-exact against the
    reference's own pairs kernels (OneSweep::DigitBinningPassPairs, Sort/OneSweep.cu:346-600) on identical input.
    Payload = element index and 20-bit keys (~1024 duplicates of every key value): any instability in either
    implementation would show as a payload mismatch."""
    n = 1 << 30
    ref = reference_case("pairs_u32_index_payload")
    assert ref["n"] == n
    k = torch.empty(n, dtype=torch.int32, device="cuda")
    v = torch.empty(n, dtype=torch.int32, device="cuda")
    g.init_random(k, 0, ref["seed"], payload=v, payload_is_index=True)
    k &= ref["key_mask"]
    assert device_digest(k) == ref["input_digest"] and device_digest(v) == ref["input_payload_digest"]
    s = g.OneSweepSorter(n, 4, 4)
    s.sort_pairs(k, v)
    assert device_digest(k) == ref["sorted_digest"], "keys differ from the reference CUDA OneSweep"
    assert device_digest(v) == ref["payload_digest"], "payloads differ from the reference CUDA OneSweep"
    # and with the reference's own payload = key input (UtilityKernels.cuh:85-117), full 32-bit keys
    ref = reference_case("pairs_u32_key_payload")
    g.init_random(k, 0, ref["seed"], payload=v)
    assert device_digest(k) == ref["input_digest"] and device_digest(v) == ref["input_payload_digest"]
    s.sort_pairs(k, v)
    s.close()
    assert device_digest(k) == ref["sorted_digest"] and device_digest(v) == ref["payload_digest"]


def test_keys_u64_2pow30(g):
    n = 1 << 30
    s = g.OneSweepSorter(n, 8, 0)
    w = torch.empty(2 * n, dtype=torch.int32, device="cuda")
    g.init_random(w, 0, 10)  # hi/lo words are consecutive draws of the reference generator
    t = w.view(torch.int64)
    h0 = s.global_histogram(t).clone()
    s.sort_keys(t)
    assert s.validate(t) == 0
    assert torch.equal(s.global_histogram(t), h0)
    s.close()
