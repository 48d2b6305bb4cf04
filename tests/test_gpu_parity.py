"""Parity of the CUDA path (through the C-ABI) with the oracle, bit-exact, on seeded inputs -- plus with the
reference's own CUDA kernels on identical inputs, through the fixtures they produced (tests/golden/).  Needs a B200: -m gpu."""
import json
import os

import numpy as np
import pytest
import torch

from tests.oraclelib import device_digest

pytestmark = pytest.mark.gpu

DEFAULT_VARIANT = 2

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_onesweep_golden.json")
PARITY_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_onesweep_parity_golden.json")


def dev_u32(a):
    return torch.from_numpy(a.view(np.int32).copy()).cuda()


def host_u32(t):
    return t.cpu().numpy().view(np.uint32)


@pytest.fixture(scope="module")
def g():
    import gpusorting_b200 as g

    return g


@pytest.fixture(scope="module")
def sorter(g):
    s = g.OneSweepSorter(1 << 22, 4, 4)
    yield s
    s.close()


def tile_keys(sorter):
    return sorter.info("tile_keys")


# ---- against the reference's own CUDA kernels ------------------------------------------------------

def test_bit_exact_vs_reference_cuda(g, sorter):
    """Keys and pairs (payload = key, as the reference generates them) against the reference's CUDA OneSweep on the
    same inputs, through device digests of its inputs and outputs (tests/golden/make_ref_golden.py)."""
    cases = json.load(open(PARITY_GOLDEN))["bit_exact"]
    assert [(c["n"], c["seed"]) for c in cases] == [(7680, 7680), (9999, 9999), (1 << 20, 10), (1 << 22, 22)]
    n = 1 << 22
    a, pa = torch.empty(n, dtype=torch.int32, device="cuda"), torch.empty(n, dtype=torch.int32, device="cuda")
    for c in cases:
        size, want = c["n"], c["keys"]
        mine = a[:size]
        g.init_random(mine, 0, c["seed"])
        assert device_digest(mine) == want["input_digest"], f"keys input n={size}"
        sorter.sort_keys(mine)
        assert device_digest(mine) == want["sorted_digest"], f"keys n={size}"
        assert want["ref_validate_errors"] == 0 and sorter.validate(mine) == 0
        mk, mv, want = a[:size], pa[:size], c["pairs"]
        g.init_random(mk, 0, c["seed"], payload=mv)
        assert device_digest(mk) == want["input_digest"] and device_digest(mv) == want["input_payload_digest"], f"pairs input n={size}"
        sorter.sort_pairs(mk, mv)
        assert device_digest(mk) == want["sorted_digest"] and device_digest(mv) == want["payload_digest"], f"pairs n={size}"


@pytest.mark.skipif(not os.path.exists(GOLDEN), reason="golden fixture not generated yet")
def test_cuda_path_reproduces_reference_golden_vectors(g, oracle):
    cases = json.load(open(GOLDEN))["cases"]
    s = g.OneSweepSorter(max(c["n"] for c in cases), 4, 4)
    for c in cases:
        n = c["n"]
        t = torch.empty(n, dtype=torch.int32, device="cuda")
        p = torch.empty(n, dtype=torch.int32, device="cuda") if c["pairs"] else None
        g.init_random(t, c["and_count"], c["seed"], payload=p)
        assert oracle.digest(host_u32(t)) == c["input_digest"]
        hist = s.global_histogram(t).cpu().numpy().astype(np.uint64)
        assert oracle.digest(hist.reshape(-1)) == c["global_hist_digest"]
        if c["pairs"]:
            s.sort_pairs(t, p)
            assert oracle.digest(host_u32(p)) == c["payload_digest"]
        else:
            s.sort_keys(t)
        assert oracle.digest(host_u32(t)) == c["sorted_digest"]
    s.close()


# ---- against the oracle ------------------------------------------------------------------------------

def test_atomic_rank_selftest_passed(sorter):
    assert sorter.info("atomic_order_ok") == 1
    assert sorter.info("rank_mode") == 0


def test_init_random_matches_oracle(g, oracle):
    for n, andc, seed in [(7680, 0, 7680), (65537, 0, 10), (1 << 20, 3, 10)]:
        t = torch.empty(n, dtype=torch.int32, device="cuda")
        g.init_random(t, andc, seed)
        assert np.array_equal(host_u32(t), oracle.init_random_u32(n, andc, seed))


@pytest.mark.parametrize("variant,small", [(0, 1), (1, 1), (2, 1), (2, 0)])
@pytest.mark.parametrize("mode", [0, 1])
def test_keys_u32_edge_sizes(sorter, oracle, mode, variant, small):
    """small = 0: n <= one tile goes through the ordinary kernels too (the single-CTA small-n path is switched off)"""
    sorter.set_option("rank_mode", mode)
    sorter.set_option("variant", variant)
    sorter.set_option("small_path", small)
    T = tile_keys(sorter)
    sizes = [0, 1, 2, 3, 31, 32, 33, 255, 256, 257, 1000, T - 1, T, T + 1, 2 * T - 1, 2 * T, 2 * T + 1, 3 * T + 17, 100003]
    try:
        for n in sizes:
            k = oracle.init_random_u32(n, 0, 1000 + n) if n else np.empty(0, np.uint32)
            t = torch.empty(max(n, 4), dtype=torch.int32, device="cuda")
            t[:n] = dev_u32(k)
            sorter.sort_keys(t, n)
            assert np.array_equal(host_u32(t[:n]), oracle.sort_keys(k)), f"n={n} mode={mode} variant={variant} small={small}"
    finally:
        sorter.set_option("rank_mode", 0)
        sorter.set_option("variant", DEFAULT_VARIANT)
        sorter.set_option("small_path", 1)


@pytest.mark.parametrize("variant,small", [(0, 1), (1, 1), (2, 1), (2, 0)])
def test_reference_size_sweep(sorter, oracle, variant, small):
    """The reference's TestAllKeysOnly sweep shape (OneSweepDispatcher.cuh:98-113): sizes across one..two of ITS
    tiles (7680..15360) and across one..two of OUR tiles, seed = n, checked bit-exactly (the reference only
    checks sortedness)."""
    T = tile_keys(sorter)
    sizes = list(range(7680, 15361, 193)) + list(range(T, 2 * T + 1, 331))
    buf = torch.empty(max(sizes), dtype=torch.int32, device="cuda")
    sorter.set_option("variant", variant)
    sorter.set_option("small_path", small)
    try:
        for n in sizes:
            k = oracle.init_random_u32(n, 0, n)
            buf[:n] = dev_u32(k)
            sorter.sort_keys(buf, n)
            assert np.array_equal(host_u32(buf[:n]), oracle.sort_keys(k)), f"n={n}"
    finally:
        sorter.set_option("variant", DEFAULT_VARIANT)
        sorter.set_option("small_path", 1)


@pytest.mark.parametrize("variant", [0, 1, 2])
@pytest.mark.parametrize("andc", [0, 1, 2, 3, 4])
def test_entropy_presets_2pow22(sorter, oracle, andc, variant):
    n = 1 << 22
    sorter.set_option("variant", variant)
    try:
        k = oracle.init_random_u32(n, andc, 10)
        t = dev_u32(k)
        sorter.sort_keys(t)
        assert np.array_equal(host_u32(t), oracle.sort_keys(k))
        assert sorter.validate(t) == 0
    finally:
        sorter.set_option("variant", DEFAULT_VARIANT)


@pytest.mark.parametrize("variant", [1, 2])
def test_adversarial_distributions(sorter, oracle, variant):
    sorter.set_option("variant", variant)
    n = 300001
    rng = np.random.default_rng(1)
    cases = {
        "all_equal": np.full(n, 0xDEADBEEF, np.uint32),
        "all_zero": np.zeros(n, np.uint32),
        "all_ones": np.full(n, 0xFFFFFFFF, np.uint32),  # collides with the tile padding value
        "sorted": np.arange(n, dtype=np.uint32),
        "reversed": np.arange(n, dtype=np.uint32)[::-1].copy(),
        "two_values": rng.integers(0, 2, n).astype(np.uint32) * np.uint32(0xFF00FF00),
        "one_digit_varies": (rng.integers(0, 256, n).astype(np.uint32) << np.uint32(16)),
        "top_byte_ff": rng.integers(0, 1 << 24, n).astype(np.uint32) | np.uint32(0xFF000000),
    }
    try:
        for name, k in cases.items():
            t = dev_u32(k)
            sorter.sort_keys(t)
            assert np.array_equal(host_u32(t), np.sort(k)), name
    finally:
        sorter.set_option("variant", DEFAULT_VARIANT)


@pytest.mark.parametrize("variant", [0, 2])
@pytest.mark.parametrize("mode", [0, 1])
def test_pairs_are_stable_payload_is_index(sorter, oracle, mode, variant):
    sorter.set_option("rank_mode", mode)
    sorter.set_option("variant", variant)
    try:
        T = tile_keys(sorter)
        for n, mask in [(1, 0xFFFFFFFF), (T + 3, 0xFF), (100003, 0xFFF), (1 << 20, 0xFFFFFFFF), (1 << 20, 0x3)]:
            k = oracle.init_random_u32(n, 0, 99 + n) & np.uint32(mask)
            v = np.arange(n, dtype=np.uint32)
            tk, tv = dev_u32(k), dev_u32(v)
            sorter.sort_pairs(tk, tv)
            wk, wv = oracle.sort_pairs(k, v)
            assert np.array_equal(host_u32(tk), wk) and np.array_equal(host_u32(tv), wv), f"n={n} mask={mask:x}"
    finally:
        sorter.set_option("rank_mode", 0)
        sorter.set_option("variant", DEFAULT_VARIANT)


@pytest.mark.parametrize("variant", [0, 1, 2])
def test_keys_u64(g, oracle, variant):
    s = g.OneSweepSorter(1 << 21, 8, 0)
    s.set_option("variant", variant)
    T = s.info("tile_keys")
    for n in [0, 1, 2, T - 1, T + 1, 5 * T + 11, 1 << 20]:
        k = oracle.init_random_u64(n, 0, 10 + n) if n else np.empty(0, np.uint64)
        t = torch.empty(max(n, 2), dtype=torch.int64, device="cuda")
        t[:n] = torch.from_numpy(k.view(np.int64).copy()).cuda()
        s.sort_keys(t, n)
        assert np.array_equal(t[:n].cpu().numpy().view(np.uint64), oracle.sort_keys(k)), f"n={n}"
    # keys that differ only in the high word
    k = (np.arange(70001, dtype=np.uint64)[::-1].copy() << np.uint64(32)) | np.uint64(7)
    t = torch.from_numpy(k.view(np.int64).copy()).cuda()
    s.sort_keys(t)
    assert np.array_equal(t.cpu().numpy().view(np.uint64), np.sort(k))
    s.close()


def test_global_histogram_kernel(sorter, oracle):
    for n in [1, 5, 4097, 1 << 20]:
        k = oracle.init_random_u32(n, 1, 4)
        h = sorter.global_histogram(dev_u32(k)).cpu().numpy().astype(np.uint64)
        assert np.array_equal(h, oracle.global_histogram(k)), f"n={n}"


def test_single_digit_binning_pass(sorter, oracle):
    n = 250007
    k = oracle.init_random_u32(n, 0, 8)
    v = np.arange(n, dtype=np.uint32)
    for shift in (0, 8, 16, 24):
        src, dst = dev_u32(k), torch.empty(n, dtype=torch.int32, device="cuda")
        sorter.digit_binning_pass(src, dst, shift)
        assert np.array_equal(host_u32(dst), oracle.binning_pass(k, shift)), f"shift={shift}"
    sv, dv = dev_u32(v), torch.empty(n, dtype=torch.int32, device="cuda")
    src, dst = dev_u32(k), torch.empty(n, dtype=torch.int32, device="cuda")
    sorter.digit_binning_pass(src, dst, 8, sv, dv)
    wk, wv = oracle.binning_pass(k, 8, v)
    assert np.array_equal(host_u32(dst), wk) and np.array_equal(host_u32(dv), wv)


@pytest.mark.parametrize("variant", [0, 1, 2])
def test_top_bits_pass_few_bins(sorter, oracle, variant):
    """A pass on the top k <= 5 bits (what the sharded exchange runs): 2..32 bins, runs of thousands of keys."""
    sorter.set_option("variant", variant)
    try:
        T = tile_keys(sorter)
        for n in (3 * T + 1234, 1 << 20, 777):
            k = oracle.init_random_u32(n, 0, 21 + n)
            for shift in (31, 29, 27, 26, 13):
                src, dst = dev_u32(k), torch.empty(n, dtype=torch.int32, device="cuda")
                sorter.digit_binning_pass(src, dst, shift)
                assert np.array_equal(host_u32(dst), oracle.binning_pass(k, shift)), f"n={n} shift={shift}"
        # skew: everything in one top bin
        k = oracle.init_random_u32(200000, 0, 5) | np.uint32(0xE0000000)
        src, dst = dev_u32(k), torch.empty(k.size, dtype=torch.int32, device="cuda")
        sorter.digit_binning_pass(src, dst, 29)
        assert np.array_equal(host_u32(dst), oracle.binning_pass(k, 29))
    finally:
        sorter.set_option("variant", DEFAULT_VARIANT)


def test_host_buffer_entry_points(g, oracle):
    s = g.OneSweepSorter(1 << 20, 4, 4)
    k = oracle.init_random_u32(1 << 20, 0, 31)
    a = k.copy()
    s.sort_host(a)
    assert np.array_equal(a, np.sort(k))
    kk, vv = (k & np.uint32(0xFFFF)).copy(), np.arange(k.size, dtype=np.uint32)
    s.sort_host(kk, vv)
    wk, wv = oracle.sort_pairs(k & np.uint32(0xFFFF), np.arange(k.size, dtype=np.uint32))
    assert np.array_equal(kk, wk) and np.array_equal(vv, wv)
    pinned = torch.from_numpy(k.view(np.int32).copy()).pin_memory()
    s.sort_host(pinned)
    assert np.array_equal(pinned.numpy().view(np.uint32), np.sort(k))
    s.close()


def test_error_behaviour(g, sorter):
    t = torch.zeros(16, dtype=torch.int32, device="cuda")
    small = g.OneSweepSorter(1024, 4, 0)
    with pytest.raises(g.OneSweepError) as e:
        small.sort_keys(torch.zeros(2048, dtype=torch.int32, device="cuda"))  # n > max_n
    assert e.value.status == -2
    small.close()
    with pytest.raises(ValueError):  # n beyond the tensor
        sorter.sort_keys(t, 17)
    with pytest.raises(g.OneSweepError):  # misaligned keys
        sorter.sort_keys(t[1:], 8)
    with pytest.raises(TypeError):
        sorter.sort_keys(torch.zeros(16, dtype=torch.float32, device="cuda"))
    with pytest.raises(g.OneSweepError):  # unknown option
        sorter.set_option("no_such_option", 1)
    ko = g.OneSweepSorter(1024, 4, 0)
    with pytest.raises(g.OneSweepError):  # keys-only sorter asked for pairs
        ko.sort_pairs(t, t.clone())
    ko.close()


def test_repeated_sorts_reuse_descriptors_without_clearing(sorter, oracle):
    """Epoch-stamped descriptors: many sorts of different sizes back to back on one handle, no memsets."""
    e0 = sorter.info("epoch")
    sizes = [50000, 1 << 20, 777, 1 << 19, 50001] * 3
    for i, n in enumerate(sizes):
        k = oracle.init_random_u32(n, i % 3, 5 + i)
        t = dev_u32(k)
        sorter.sort_keys(t)
        assert np.array_equal(host_u32(t), oracle.sort_keys(k))
    # one epoch per DigitBinningPass launch; a sort of at most one tile takes the single-CTA path and launches none
    assert sorter.info("epoch") == e0 + 4 * sum(n > sorter.info("small_path_max_n") for n in sizes)


def test_sort_on_side_stream_and_module_level_Sort(g, oracle):
    k = oracle.init_random_u32(1 << 18, 0, 3)
    st = torch.cuda.Stream()
    t = dev_u32(k)
    torch.cuda.synchronize()
    with torch.cuda.stream(st):
        g.Sort(t, stream=st)
    st.synchronize()
    assert np.array_equal(host_u32(t), np.sort(k))
    tk, tv = dev_u32(k & np.uint32(0xFF)), dev_u32(np.arange(k.size, dtype=np.uint32))
    g.Sort(tk, tv)
    assert np.array_equal(host_u32(tv), np.argsort(k & np.uint32(0xFF), kind="stable").astype(np.uint32))


def test_dispatcher_mirror_runs_reference_tests(g):
    d = g.OneSweepDispatcher(True, 1 << 20)
    passed, total = d.TestAllKeysOnly(small_step=509, large_exps=(20,))
    assert passed == total and total > 10
    assert d.BatchTimingKeysOnly(1 << 20, 3, 10, g.ENTROPY_PRESET_1) > 0
    p = g.OneSweepDispatcher(False, 1 << 20)
    passed, total = p.TestAllPairs(small_step=997, large_exps=(20,))
    assert passed == total
    with pytest.raises(ValueError):
        d.BatchTimingPairs(1 << 20, 1, 10)


def test_cli_runs_the_reference_protocol():
    """The C++ driver that restates the reference's main (GPUSortingCUDA.cu:16-57: TestAll sweeps + BatchTiming) on top
    of include/OneSweepB200.hpp: coarse sweep, 2^20 timing."""
    import subprocess

    exe = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpusorting_b200", "lib", "onesweep_b200_cli")
    if not os.path.exists(exe):
        pytest.skip("onesweep_b200_cli not built (make -C gpusorting_b200/csrc cli)")
    r = subprocess.run([exe, "20", "3", "257", "22"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.count("All tests passed.") == 2 and r.stdout.count("Estimated speed") == 2
