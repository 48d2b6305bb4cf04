"""SURVEY 8f ranks 2-3: entropy robustness, device-side pass skipping, begin_bit/end_bit sorts, and the forward-progress
fallback of the chained scan (reference: UtilityKernels.cuh:42-52,70-81 entropy presets; GPUSortingD3D12/Tests.h:383-393;
Sort/EmulatedDeadlocking.cu:159-267,339-345).  Bit-exact against numpy stable sorts.  -m gpu"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def dev(a):
    return torch.from_numpy(a.view(np.int32 if a.dtype.itemsize == 4 else np.int64).copy()).cuda()


def host(t, dtype=np.uint32):
    return t.cpu().numpy().view(dtype)


@pytest.fixture(scope="module")
def g():
    import gpusorting_b200 as g

    return g


@pytest.fixture()
def sorter(g):
    s = g.OneSweepSorter(1 << 21, 4, 4)
    yield s
    s.close()


CONST_CASES = [
    # (name, and-mask, or-mask, expected skip mask, expected executed passes)
    ("all_bytes_vary", 0xFFFFFFFF, 0x00000000, 0b0000, 4),
    ("low_16_bits_vary", 0x0000FFFF, 0xABCD0000, 0b1100, 2),
    ("only_byte_1_varies", 0x0000FF00, 0x12340056, 0b1101, 1),   # odd: the result must be copied back
    ("bytes_0_1_2_vary", 0x00FFFFFF, 0x7F000000, 0b1000, 3),     # odd
    ("only_top_byte_varies", 0xFF000000, 0x00000000, 0b0111, 1),
    ("all_equal", 0x00000000, 0xDEADBEEF, 0b1111, 0),
]


@pytest.mark.parametrize("name,andm,orm,skip,executed", CONST_CASES)
@pytest.mark.parametrize("n", [5, 16384 * 3 + 77, 1 << 20])
def test_passes_with_a_constant_digit_are_skipped(g, sorter, oracle, name, andm, orm, skip, executed, n):
    k = (oracle.init_random_u32(n, 0, 77 + n) & np.uint32(andm)) | np.uint32(orm)
    # the device plan belongs to the multi-kernel path: keep n <= one tile on it too (the single-CTA path has no plan)
    sorter.set_option("small_path", 0)
    try:
        t = dev(k)
        sorter.sort_keys(t)
        assert np.array_equal(host(t), np.sort(k)), name
        assert sorter.info("last_skip_mask") == skip and sorter.info("last_executed_passes") == executed
        # pairs: stability must survive skipping and the copy-back
        v = np.arange(n, dtype=np.uint32)
        tk, tv = dev(k), dev(v)
        sorter.sort_pairs(tk, tv)
        order = np.argsort(k, kind="stable")
        assert np.array_equal(host(tk), k[order]) and np.array_equal(host(tv), v[order]), name
        assert sorter.info("last_executed_passes") == executed
    finally:
        sorter.set_option("small_path", 1)


def test_short_circuit_can_be_switched_off(g, sorter, oracle):
    n = 200003
    k = oracle.init_random_u32(n, 0, 3) & np.uint32(0xFFFF)
    sorter.set_option("short_circuit", 0)
    t = dev(k)
    sorter.sort_keys(t)
    assert np.array_equal(host(t), np.sort(k))
    assert sorter.info("last_skip_mask") == 0 and sorter.info("last_executed_passes") == 4
    # histogram + scan + per place the pass and its HOT twin (one of the two returns at once)
    assert sorter.info("launches_per_sort") == 10
    sorter.set_option("hot_passes", 0)
    assert sorter.info("launches_per_sort") == 6
    sorter.set_option("hot_passes", 1)
    sorter.set_option("short_circuit", 1)
    assert sorter.info("launches_per_sort") == 12  # + copy-back of keys and values (pairs-capable handle)


@pytest.mark.parametrize("andc", [0, 1, 2, 3, 4])
def test_entropy_presets_with_skipping_u64(g, oracle, andc):
    """Thearling-Smith presets on 64-bit keys whose high word is constant: 4 of the 8 passes are skipped."""
    n = (1 << 19) + 123
    lo = oracle.init_random_u32(n, andc, 10).astype(np.uint64)
    k = lo | (np.uint64(0x00C0FFEE) << np.uint64(32))
    s = g.OneSweepSorter(n, 8, 0)
    t = dev(k)
    s.sort_keys(t)
    assert np.array_equal(host(t, np.uint64), np.sort(k))
    assert s.info("last_skip_mask") & 0xF0 == 0xF0
    s.close()


@pytest.mark.parametrize("kind,desc", [("i32", False), ("i32", True), ("f32", False), ("f32", True)])
def test_typed_keys_when_the_first_or_last_pass_is_skipped(g, sorter, kind, desc):
    """The encode/decode of typed keys happens in the first/last EXECUTED pass, whichever those are."""
    rng = np.random.default_rng(5)
    n = 100000
    if kind == "i32":
        vals = rng.integers(0, 200, n).astype(np.int32)  # bytes 1..3 of the encoded key are constant: ONE pass encodes and decodes
        bits = vals.view(np.uint32)
        order = np.argsort(-vals.astype(np.int64) if desc else vals, kind="stable")
    else:
        vals = (rng.integers(1, 256, n).astype(np.float32) * np.float32(2.0 ** -10))  # low mantissa byte is zero: pass 0 is skipped
        bits = vals.view(np.uint32)
        enc = np.where(bits >> 31 != 0, ~bits, bits | np.uint32(0x80000000))
        order = np.argsort(~enc if desc else enc, kind="stable")
    t = dev(bits.copy())
    sorter.sort_keys_typed(t, kind, desc)
    assert np.array_equal(host(t), bits[order])
    assert sorter.info("last_skip_mask") != 0
    tv = dev(np.arange(n, dtype=np.uint32))
    t = dev(bits.copy())
    sorter.sort_pairs_typed(t, tv, kind, desc)
    assert np.array_equal(host(t), bits[order]) and np.array_equal(host(tv), order.astype(np.uint32))


BIT_RANGES = [(0, 32), (0, 8), (8, 16), (0, 16), (4, 20), (3, 14), (0, 1), (31, 32), (5, 32), (0, 27), (13, 13), (9, 29)]


@pytest.mark.parametrize("begin,end", BIT_RANGES)
def test_sort_bits_u32(g, sorter, oracle, begin, end):
    for n in (1000, 16384 * 2 + 5, 1 << 20):
        k = oracle.init_random_u32(n, 0, begin * 37 + end + n)
        v = np.arange(n, dtype=np.uint32)
        mask = np.uint32((1 << (end - begin)) - 1) if end - begin < 32 else np.uint32(0xFFFFFFFF)
        order = np.argsort((k >> np.uint32(begin)) & mask, kind="stable")
        tk, tv = dev(k), dev(v)
        sorter.sort_bits(tk, begin, end, tv)
        assert np.array_equal(host(tk), k[order]) and np.array_equal(host(tv), v[order]), f"pairs n={n}"
        tk = dev(k)
        sorter.sort_bits(tk, begin, end)
        assert np.array_equal(host(tk), k[order]), f"keys n={n}"  # keys-only: the stable answer is THE answer for whole keys


@pytest.mark.parametrize("begin,end", [(0, 64), (0, 40), (17, 49), (32, 64), (60, 64), (7, 8)])
def test_sort_bits_u64(g, oracle, begin, end):
    n = (1 << 18) + 99
    k = oracle.init_random_u64(n, 0, begin + end)
    s = g.OneSweepSorter(n, 8, 0)
    mask = np.uint64((1 << (end - begin)) - 1) if end - begin < 64 else np.uint64(0xFFFFFFFFFFFFFFFF)
    order = np.argsort((k >> np.uint64(begin)) & mask, kind="stable")
    t = dev(k)
    s.sort_bits(t, begin, end)
    assert np.array_equal(host(t, np.uint64), k[order])
    s.close()


def test_sort_bits_rejects_bad_ranges(g, sorter):
    t = torch.zeros(64, dtype=torch.int32, device="cuda")
    for b, e in [(-1, 8), (0, 33), (9, 8)]:
        with pytest.raises(g.OneSweepError):
            sorter.sort_bits(t, b, e)


@pytest.mark.parametrize("n", [5000, 16384 * 3 + 77])
def test_misaligned_payloads_are_rejected(g, sorter, n):
    """Payloads must be 16-byte aligned like the keys: after an odd number of executed passes the copy-back moves them
    in 16-byte words.  Keys below 2^24 skip the top byte's pass (3 executed) -- the case a misaligned payload would fault
    in -- and the small-n path (n = 5000) refuses it too, so acceptance does not depend on n.  A refused call leaves both
    buffers untouched, and the handle sorts correctly afterwards."""
    k = (np.random.default_rng(n).integers(0, 1 << 24, n)).astype(np.uint32)
    tk = dev(k)
    storage = torch.arange(n + 1, dtype=torch.int32, device="cuda")
    tv = storage[1:]  # contiguous, 4-byte aligned only
    assert tv.data_ptr() % 16 == 4
    v0 = tv.clone()
    calls = [lambda: sorter.sort_pairs(tk, tv), lambda: sorter.sort_bits(tk, 0, 24, tv),
             lambda: sorter.sort_pairs_typed(tk, tv, "i32", True)]
    for call in calls:
        with pytest.raises(g.OneSweepError) as e:
            call()
        assert e.value.status == -1
        assert np.array_equal(host(tk), k) and torch.equal(tv, v0), "a refused sort must not touch the buffers"
    tv = torch.arange(n, dtype=torch.int32, device="cuda")
    sorter.sort_pairs(tk, tv)
    order = np.argsort(k, kind="stable")
    assert np.array_equal(host(tk), k[order]) and np.array_equal(host(tv), order.astype(np.uint32))
    if n > sorter.info("small_path_max_n"):
        assert sorter.info("last_skip_mask") == 0b1000 and sorter.info("last_executed_passes") == 3


@pytest.mark.parametrize("stall_every", [1, 2, 5])
def test_lookback_fallback_rereduces_stalled_tiles(g, oracle, stall_every):
    """Forward-progress fallback (EmulatedDeadlocking.cu:159-267; test hook as :339-345): every N-th tile WITHHOLDS its
    reduction, so its successors hit the spin cap and must re-reduce it themselves.  Output stays bit-exact."""
    n = 16384 * 23 + 4321
    s = g.OneSweepSorter(n, 4, 4)
    s.set_option("spin_cap", 16)
    s.set_option("debug_stall_every", stall_every)
    for andc, seed in [(0, 1), (3, 2)]:
        k = oracle.init_random_u32(n, andc, seed)
        t = dev(k)
        s.sort_keys(t)
        assert np.array_equal(host(t), oracle.sort_keys(k)), f"keys stall_every={stall_every}"
        v = np.arange(n, dtype=np.uint32)
        tk, tv = dev(k & np.uint32(0xFFF)), dev(v)
        s.sort_pairs(tk, tv)
        wk, wv = oracle.sort_pairs(k & np.uint32(0xFFF), v)
        assert np.array_equal(host(tk), wk) and np.array_equal(host(tv), wv)
    # typed keys: the re-reduction must count digits of the ENCODED keys in the first pass
    f = (np.random.default_rng(0).standard_normal(n) * 100).astype(np.float32)
    t = dev(f.view(np.uint32).copy())
    s.sort_keys_typed(t, "f32")
    assert np.array_equal(host(t).view(np.float32), np.sort(f))
    s.close()


def test_u64_fallback(g, oracle):
    n = 8192 * 9 + 17
    s = g.OneSweepSorter(n, 8, 0)
    s.set_option("spin_cap", 8)
    s.set_option("debug_stall_every", 3)
    k = oracle.init_random_u64(n, 0, 4)
    t = dev(k)
    s.sort_keys(t)
    assert np.array_equal(host(t, np.uint64), np.sort(k))
    s.close()


@pytest.mark.parametrize("andc", [2, 3, 4])
def test_hot_passes_low_entropy_keys_and_pairs(g, oracle, andc):
    """Entropy presets 3-5 (UtilityKernels.cuh:42-52): one bin holds 34-78 % of every digit place, the Scan kernel flags
    the passes hot and the HOT instantiation of the DigitBinningPass (one ballot per round for the tile's most frequent
    digit) executes them; same results as the plain kernel and the oracle, stable for pairs."""
    n = (1 << 22) + 4099
    k = oracle.init_random_u32(n, andc, 5)
    v = np.arange(n, dtype=np.uint32)
    wk, wv = oracle.sort_pairs(k, v)
    with g.OneSweepSorter(n, 4, 4) as s:
        for hot in (1, 0):
            s.set_option("hot_passes", hot)
            t = dev(k)
            s.sort_keys(t)
            assert np.array_equal(host(t), wk)
            assert (s.info("last_hot_mask") != 0) == bool(hot)
            tk, tv = dev(k), dev(v)
            s.sort_pairs(tk, tv)
            assert np.array_equal(host(tk), wk) and np.array_equal(host(tv), wv)
    with g.OneSweepSorter(n, 8, 0) as s8:  # 64-bit keys: the low word is low-entropy, the high word uniform
        k8 = k.astype(np.uint64) | (oracle.init_random_u32(n, 0, 6).astype(np.uint64) << np.uint64(32))
        t = dev(k8)
        s8.sort_keys(t)
        assert np.array_equal(host(t, np.uint64), np.sort(k8))
        assert s8.info("last_hot_mask") & 0x0F == 0x0F and s8.info("last_hot_mask") & 0xF0 == 0
