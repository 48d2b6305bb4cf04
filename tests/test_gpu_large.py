"""Exact answers at full size and past 32-bit element indices.

* 2^28 keys: the output is compared element by element with torch.sort(stable=True) of the radix key (tests/sortcheck)
  -- 64-bit keys (uniform and entropy preset 4, which runs HOT), preset-4 u32 keys and pairs, descending float pairs
  with heavy ties, a bit-range sort with a 5-bit last digit, and pairs in ballot rank mode.
* n = 2^32 + 4099 keys, 2^31 + 4099 pairs and 2^31 + 17 64-bit keys (the interface takes a 64-bit n, up to 2^34):
  too large for a second sort to compare with, so they are certified by tests/sortcheck -- sorted, a permutation that
  carries every key's origin, equal keys in input order, or for keys only sorted plus the exact multiset.

Every sort runs once.  The 2^28 cases need ~15-17 GiB of device memory and the larger ones tens of GB; on a shared GPU
each case skips, saying so, when that much is not free.  The HOT cases pin the atomic rank mode (see test_gpu_paths).  -m gpu"""
import numpy as np
import pytest
import torch

from tests.sortcheck import bincount_chunked, certify_sorted_multiset, certify_stable_sort, radix_key_torch
from tests.test_gpu_paths import atomic_rank_mode

pytestmark = pytest.mark.gpu

GiB = 1 << 30
CHUNK = 1 << 27


@pytest.fixture(scope="module")
def g():
    import gpusorting_b200 as g

    return g


@pytest.fixture(autouse=True)
def release_memory():
    yield
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def require_free(nbytes, what):
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes + 2 * GiB:
        pytest.skip(f"{what} needs ~{nbytes / GiB:.0f} GiB of device memory, {free / GiB:.0f} GiB are free on this shared GPU")
    torch.cuda.reset_peak_memory_stats()


def report_peak(g, what, n, key_bytes, value_bytes):
    peak = torch.cuda.max_memory_allocated() + g.lib.osb200_workspace_bytes(n, key_bytes, value_bytes)
    print(f"{what}: peak device memory {peak / GiB:.1f} GiB (tensors + sorter workspace)")


def stable_order(bits, kind="u", desc=False, begin=0, end=None):
    return torch.sort(radix_key_torch(bits, kind, desc, begin, end), stable=True)[1]


def to_int32(x):
    """int64 values in [0, 2^32) -> the int32 with the same bits"""
    return torch.where(x >= 1 << 31, x - (1 << 32), x).to(torch.int32)


# ---- 2^28, element by element -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("and_count", [0, 3])
def test_u64_keys_2pow28_exact(g, and_count):
    n = 1 << 28
    require_free(n * 72, "2^28 u64 keys")
    w = torch.empty(2 * n, dtype=torch.int32, device="cuda")
    g.init_random(w, and_count, 101 + and_count)
    t = w.view(torch.int64)
    want = t[stable_order(t)]
    with g.OneSweepSorter(n, 8, 0) as s:
        if and_count:
            atomic_rank_mode(s)
        s.sort_keys(t)
        hot = s.info("last_hot_mask")
    assert torch.equal(t, want)
    assert (hot == 0xFF) if and_count else (hot == 0)
    report_peak(g, "2^28 u64 keys", n, 8, 0)


def test_u32_keys_and_pairs_2pow28_preset4_hot(g):
    n = 1 << 28
    require_free(n * 64, "2^28 u32 keys and pairs")
    k = torch.empty(n, dtype=torch.int32, device="cuda")
    v = torch.empty(n, dtype=torch.int32, device="cuda")
    g.init_random(k, 3, 102, payload=v, payload_is_index=True)
    order = stable_order(k)
    want = k[order]
    with g.OneSweepSorter(n, 4, 4) as s:
        atomic_rank_mode(s)
        t = k.clone()
        s.sort_keys(t)
        assert s.info("last_hot_mask") == 0b1111
        assert torch.equal(t, want), "keys"
        del t
        s.sort_pairs(k, v)
        assert s.info("last_hot_mask") == 0b1111
    assert torch.equal(k, want), "pairs: keys"
    assert torch.equal(v.to(torch.int64), order), "pairs: payload order"
    report_peak(g, "2^28 u32 keys and pairs", n, 4, 4)


def test_f32_descending_pairs_2pow28_heavy_ties(g):
    n = 1 << 28
    require_free(n * 64, "2^28 f32 pairs")
    k = torch.empty(n, dtype=torch.int32, device="cuda")
    g.init_random(k, 0, 103)
    f = ((k & 0xFFF) - 2048).to(torch.float32) * 0.25  # 4,096 values, both signs and +0: ~65,000 copies of each
    f[::1000] = -0.0
    bits = f.view(torch.int32)
    del k, f
    order = stable_order(bits, "f", True)
    want = bits[order]
    v = torch.arange(n, dtype=torch.int32, device="cuda")
    with g.OneSweepSorter(n, 4, 4) as s:
        s.sort_pairs_typed(bits, v, "f32", descending=True)
    assert torch.equal(bits, want), "keys"
    assert torch.equal(v.to(torch.int64), order), "payload order (ties must keep their input order)"
    report_peak(g, "2^28 f32 pairs", n, 4, 4)


def test_sort_bits_0_29_pairs_2pow28(g):
    n = 1 << 28
    require_free(n * 64, "2^28 bit-range pairs")
    k = torch.empty(n, dtype=torch.int32, device="cuda")
    g.init_random(k, 0, 104)
    order = stable_order(k, begin=0, end=29)
    want = k[order]
    v = torch.arange(n, dtype=torch.int32, device="cuda")
    with g.OneSweepSorter(n, 4, 4) as s:
        s.sort_bits(k, 0, 29, v)
    assert torch.equal(k, want) and torch.equal(v.to(torch.int64), order)
    report_peak(g, "2^28 bit-range pairs", n, 4, 4)


def test_pairs_2pow28_ballot_rank_mode(g):
    n = 1 << 28
    require_free(n * 64, "2^28 ballot-ranked pairs")
    k = torch.empty(n, dtype=torch.int32, device="cuda")
    v = torch.empty(n, dtype=torch.int32, device="cuda")
    g.init_random(k, 0, 105, payload=v, payload_is_index=True)
    k &= 0xFFFFF  # ~256 copies of every key
    order = stable_order(k)
    want = k[order]
    with g.OneSweepSorter(n, 4, 4) as s:
        s.set_option("rank_mode", 1)
        assert s.info("rank_mode") == 1
        s.sort_pairs(k, v)
    assert torch.equal(k, want) and torch.equal(v.to(torch.int64), order)
    report_peak(g, "2^28 ballot-ranked pairs", n, 4, 4)


# ---- past 2^31 and 2^32 elements, certified ---------------------------------------------------------------------------
def test_u32_keys_past_2pow32_certified(g):
    """key = (x * C) mod 2^32 for a 24-bit generator value x: every byte varies, so all four passes run; multiplying by
    C^-1 gives x back, so the multiset check is an exact 2^24-bin count of input against output."""
    n = (1 << 32) + 4099
    require_free(n * 4 + g.lib.osb200_workspace_bytes(n, 4, 0) + 6 * CHUNK * 8, "2^32 + 4099 keys")
    C = 0x9E3779B1
    CINV = pow(C, -1, 1 << 32)
    k = torch.empty(n, dtype=torch.int32, device="cuda")
    g.init_random(k, 0, 106)
    for s0 in range(0, n, CHUNK):
        x = k[s0:s0 + CHUNK].to(torch.int64) & 0xFFFFFF
        k[s0:s0 + CHUNK] = to_int32((x * C) & 0xFFFFFFFF)
    del x
    bin_of = lambda t: ((t.to(torch.int64) & 0xFFFFFFFF) * CINV) & 0xFFFFFFFF  # noqa: E731  (x back)
    in_counts = bincount_chunked(k, bin_of, 1 << 24, CHUNK)
    with g.OneSweepSorter(n, 4, 0) as s:
        hist = s.global_histogram(k)
        want = torch.zeros(4, 256, dtype=torch.int64, device="cuda")
        for s0 in range(0, n, CHUNK):
            u = k[s0:s0 + CHUNK].to(torch.int64) & 0xFFFFFFFF
            for p in range(4):
                want[p] += torch.bincount((u >> (8 * p)) & 255, minlength=256)
        del u
        assert torch.equal(hist, want), "global histogram"
        assert int(want.sum()) == 4 * n and bool(((want > 0).sum(dim=1) > 1).all())
        s.sort_keys(k)
        assert s.info("last_skip_mask") == 0 and s.info("last_executed_passes") == 4
    certify_sorted_multiset(in_counts, k, bin_of, chunk=CHUNK)
    report_peak(g, "u32 keys, n = 2^32 + 4099", n, 4, 0)


def test_u32_pairs_past_2pow31_certified(g):
    """payload = index (beyond 2^31, still 32 bits); 20-bit keys, ~2,000 copies of each: the top byte's pass is skipped,
    three passes execute and the copy-back moves 2^31 payloads"""
    n = (1 << 31) + 4099
    require_free(3 * n * 4 + n + g.lib.osb200_workspace_bytes(n, 4, 4) + 8 * CHUNK * 8, "2^31 + 4099 pairs")
    k = torch.empty(n, dtype=torch.int32, device="cuda")
    v = torch.empty(n, dtype=torch.int32, device="cuda")
    g.init_random(k, 0, 107, payload=v, payload_is_index=True)
    k &= 0xFFFFF
    kin = k.clone()
    with g.OneSweepSorter(n, 4, 4) as s:
        s.sort_pairs(k, v)
        assert s.info("last_skip_mask") == 0b1000 and s.info("last_executed_passes") == 3
    certify_stable_sort(kin, k, v, chunk=CHUNK)
    report_peak(g, "u32 pairs, n = 2^31 + 4099", n, 4, 4)


def test_u64_keys_past_2pow31_certified(g):
    """key = (hi << 32) | index with a preset-4 hi word (the high passes run HOT): the whole-key sort is the stable sort
    on hi, and the low words are the payload that certifies it"""
    n = (1 << 31) + 17
    require_free(n * 8 + n * 4 + n + g.lib.osb200_workspace_bytes(n, 8, 0) + 8 * CHUNK * 8, "2^31 + 17 64-bit keys")
    hi = torch.empty(n, dtype=torch.int32, device="cuda")
    g.init_random(hi, 3, 108)
    t = torch.empty(n, dtype=torch.int64, device="cuda")
    for s0 in range(0, n, CHUNK):
        e = min(s0 + CHUNK, n)
        t[s0:e] = (hi[s0:e].to(torch.int64) << 32) | torch.arange(s0, e, dtype=torch.int64, device="cuda")
    with g.OneSweepSorter(n, 8, 0) as s:
        atomic_rank_mode(s)
        s.sort_keys(t)
        hot = s.info("last_hot_mask")
    assert hot & 0xF0 == 0xF0, f"hot mask {hot:#x}"
    words = t.view(torch.int32)  # little-endian: [lo, hi] per key
    certify_stable_sort(hi, words[1::2], words[0::2], chunk=CHUNK)
    report_peak(g, "u64 keys, n = 2^31 + 17", n, 8, 0)
