"""The oracle (oracle/oracle.c) against numpy and against the golden fixtures produced by the reference's own
CUDA kernels (tests/golden/ref_onesweep_golden.json).  Runs on CPU."""
import json
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_onesweep_golden.json")


def test_generator_known_values(oracle):
    # InitRandom(seed=10, andCount=0): values pinned by the reference kernel run recorded in the golden file
    k = oracle.init_random_u32(1 << 17, 0, 10)
    assert [hex(x) for x in k[:4]] == ["0xffeb2900", "0x88b92968", "0x11876dd0", "0x9a57ca38"]
    assert [hex(x) for x in k[65536:65538]] == ["0x145cb47f", "0x6766deee"]


def test_generator_entropy_presets_and(oracle):
    # AND-ing more draws can only clear bits; population count must fall monotonically (Thearling-Smith)
    pops = []
    for andc in range(5):
        k = oracle.init_random_u32(1 << 16, andc, 10)
        pops.append(int(np.unpackbits(k.view(np.uint8)).sum()))
    assert all(a > b for a, b in zip(pops, pops[1:]))
    assert abs(pops[0] / (32 * (1 << 16)) - 0.5) < 0.01


@pytest.mark.parametrize("n", [0, 1, 2, 255, 256, 257, 7680, 7681, 100003, 1 << 20])
def test_sort_keys_u32_matches_numpy(oracle, n):
    k = oracle.init_random_u32(n, 0, 10 + n) if n else np.empty(0, np.uint32)
    assert np.array_equal(oracle.sort_keys(k), np.sort(k, kind="stable"))


@pytest.mark.parametrize("andc", [0, 2, 4])
def test_sort_pairs_is_stable(oracle, andc):
    n = 200003
    k = oracle.init_random_u32(n, andc, 77) & np.uint32(0x3FF)  # many duplicate keys
    v = np.arange(n, dtype=np.uint32)
    sk, sv = oracle.sort_pairs(k, v)
    order = np.argsort(k, kind="stable").astype(np.uint32)
    assert np.array_equal(sv, order) and np.array_equal(sk, k[order])
    # std::stable_sort baseline agrees
    k2, v2 = k.copy(), v.copy()
    oracle.lib.orc_std_stable_sort_pairs_u32(k2.ctypes.data, v2.ctypes.data, n)
    assert np.array_equal(k2, sk) and np.array_equal(v2, sv)


def test_sort_keys_u64_matches_numpy(oracle):
    k = oracle.init_random_u64(150001, 0, 10)
    assert np.array_equal(oracle.sort_keys(k), np.sort(k))
    assert len(np.unique(k >> np.uint64(32))) > 100000  # hi words are independent draws


def test_histogram_scan_and_single_pass(oracle):
    k = oracle.init_random_u32(123457, 0, 5)
    h = oracle.global_histogram(k)
    for p in range(4):
        assert np.array_equal(h[p], np.bincount((k >> (8 * p)) & 255, minlength=256).astype(np.uint64))
    ex = oracle.scan_exclusive(h)
    assert np.array_equal(ex[2], np.concatenate([[0], np.cumsum(h[2])[:-1]]).astype(np.uint64))
    out = oracle.binning_pass(k, 8)
    order = np.argsort((k >> 8) & 255, kind="stable")
    assert np.array_equal(out, k[order])


def test_parallel_port_equals_serial(oracle):
    k = oracle.init_random_u32(1 << 20, 0, 3)
    want = oracle.sort_keys(k)
    for threads in (1, 3, 0):
        got = k.copy()
        assert oracle.sort_parallel_inplace(got, threads=threads) == 0
        assert np.array_equal(got, want)
    v = np.arange(k.size, dtype=np.uint32)
    kk, vv = (k & np.uint32(0xFFF)).copy(), v.copy()
    oracle.sort_parallel_inplace(kk, vv, threads=0)
    assert np.array_equal(vv, np.argsort(k & np.uint32(0xFFF), kind="stable").astype(np.uint32))


def test_validate_counts_inversions(oracle):
    k = np.array([1, 2, 2, 5, 4, 4, 9, 0], np.uint32)
    assert oracle.validate(k) == 2
    assert oracle.validate(np.sort(k)) == 0
    std = k.copy()
    oracle.lib.orc_std_sort_u32(std.ctypes.data, std.size)
    assert np.array_equal(std, np.sort(k))


@pytest.mark.skipif(not os.path.exists(GOLDEN), reason="golden fixture not generated yet")
def test_oracle_reproduces_reference_golden_vectors(oracle):
    """Pins the oracle to the reference: inputs, sorted outputs, payloads and histograms produced by the
    reference's own CUDA kernels on the B200 (see tests/golden/make_ref_golden.py)."""
    cases = json.load(open(GOLDEN))["cases"]
    assert len(cases) >= 10
    for c in cases:
        n = c["n"]
        k = oracle.init_random_u32(n, c["and_count"], c["seed"])
        assert [int(x) for x in k[:8]] == c["input_head"]
        assert oracle.digest(k) == c["input_digest"]
        assert c["ref_validate_errors"] == 0
        if c["pairs"]:
            sk, sv = oracle.sort_pairs(k, k.copy())  # the reference sets payload = key
            assert oracle.digest(sv) == c["payload_digest"]
        else:
            sk = oracle.sort_keys(k)
        assert [int(x) for x in sk[:8]] == c["sorted_head"]
        assert [int(x) for x in sk[-8:]] == c["sorted_tail"]
        assert oracle.digest(sk) == c["sorted_digest"]
        assert oracle.digest(oracle.global_histogram(k).reshape(-1)) == c["global_hist_digest"]


def test_oracle_reproduces_reference_parity_digests(oracle):
    """The device digests the reference produced for the GPU parity tests (tests/golden/make_ref_golden.py), recomputed
    on the CPU from the oracle: pins the fixture and oraclelib.device_digest, whatever device it runs on."""
    import torch

    from tests.oraclelib import device_digest

    cases = json.load(open(os.path.join(os.path.dirname(GOLDEN), "ref_onesweep_parity_golden.json")))["bit_exact"]
    assert len(cases) == 4
    for c in cases:
        k = oracle.init_random_u32(c["n"], 0, c["seed"])
        sk, sv = oracle.sort_pairs(k, k.copy())
        assert device_digest(torch.from_numpy(k.view(np.int32))) == c["keys"]["input_digest"] == c["pairs"]["input_digest"]
        assert device_digest(torch.from_numpy(sk.view(np.int32))) == c["keys"]["sorted_digest"] == c["pairs"]["sorted_digest"]
        assert device_digest(torch.from_numpy(sv.view(np.int32))) == c["pairs"]["payload_digest"]
