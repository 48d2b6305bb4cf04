"""The HOT instantiation of the DigitBinningPass together with the features it carries: typed keys, pass skipping and the
copy-back, bit ranges (with the <= 5-bit few-bins scatter), the forward-progress fallback, ballot ranking, and every kind
of tile (a tile-wide hot digit, a per-tile one, none, a tie, the padded last tile).

A pass is HOT when the global histogram of its digit place has a bin with >= n/8 keys and n >= 2^22 (the Scan kernel's
rule), so every case here sorts 2^22 + 4099 keys (ragged last tile for every tile size) or 2^23 + 1.  Each case compares
keys and payloads (payload = input index) bit for bit with numpy's stable argsort of the radix key, and asserts the
device plan -- skipped, hot and executed passes, exactly as tests/sortcheck.expected_plan predicts from the input --
and the rank mode it targets, so that neither a change of the heuristics nor the create-time fallback to ballot ranking
can quietly turn a case into a test of another path.  Float keys below 2^22 (NaNs of both signs, +-0, denormals) close
the file.  -m gpu"""
import numpy as np
import pytest
import torch

from tests.sortcheck import expected_plan, radix_key, stable_order

pytestmark = pytest.mark.gpu

SIZES = [(1 << 22) + 4099, (1 << 23) + 1]
W32, W64 = 0x3C5A7E11, 0x3C5A7E11D2B49687  # the tile-wide hot key of the mixed input: a different digit in every place

F32_SPECIALS = np.array([
    0x00000000, 0x80000000,              # +0, -0
    0x3F800000, 0xBF800000,              # +1, -1
    0x7F800000, 0xFF800000,              # +inf, -inf
    0x00000001, 0x00400000, 0x807FFFFF,  # denormals
    0x7FC00000, 0x7FC00001, 0xFFC00000, 0xFFC12345,  # quiet NaNs, both signs, different payloads
    0x7F800001, 0x7FA00000, 0xFF800001, 0xFFBFFFFF,  # signalling NaNs
], dtype=np.uint32)
F64_SPECIALS = np.array([
    0x0000000000000000, 0x8000000000000000, 0x3FF0000000000000, 0xBFF0000000000000,
    0x7FF0000000000000, 0xFFF0000000000000, 0x0000000000000001, 0x0008000000000000, 0x800FFFFFFFFFFFFF,
    0x7FF8000000000000, 0x7FF8000000000001, 0xFFF8000000000000, 0xFFF80000DEADBEEF,
    0x7FF0000000000001, 0x7FF4000000000000, 0xFFF0000000000001, 0xFFF7FFFFFFFFFFFF,
], dtype=np.uint64)


# ---- inputs (numpy bits; every generator is seeded) ----------------------------------------------------------------
def low_entropy(oracle, n, width, seed):
    """L: the reference's entropy preset 4 (AND of 4 draws): one bin holds ~60 % of every digit place"""
    return oracle.init_random_u32(n, 3, seed) if width == 32 else oracle.init_random_u64(n, 3, seed)


def mixed(n, width, seed):
    """M: per 16,384-key tile (= two 8,192-key tiles of pairs / 64-bit keys, which then come in identical pairs), six
    kinds in turn -- 70 % one tile-wide key W (the hot digit of the whole pass), 70 % a key that changes per tile, no
    dominant key at all, W again, an exact half/half tie of two keys that differ in every digit, W again.  The padded last
    tile is dominated by the all-ones padding digit."""
    dt = np.uint32 if width == 32 else np.uint64
    rng = np.random.default_rng(seed)
    top = np.iinfo(dt).max
    out = rng.integers(0, top, n, dtype=dt, endpoint=True)
    unit = 8192
    for b in range((n + unit - 1) // unit):
        seg = out[b * unit:(b + 1) * unit]
        m, t16 = seg.size, b // 2
        kind = t16 % 6
        if kind in (0, 3, 5):
            seg[rng.random(m) < 0.7] = W32 if width == 32 else W64
        elif kind == 1:
            seg[rng.random(m) < 0.7] = dt((t16 * 0x9E3779B97F4A7C15 + seed) & top)
        elif kind == 4:
            a = dt((t16 * 0xD1B54A32D192ED03 + 1) & top)
            half = rng.permutation(m) < m // 2
            seg[half] = a
            seg[~half] = a ^ dt(0xA5A5A5A5A5A5A5A5 & top)
    return out


def floats(n, width, seed):
    """F: 70 % special values (+-0, +-1, +-inf, denormals, quiet and signalling NaNs of both signs and several
    payloads), 30 % random bit patterns; built as integers so the NaN payloads survive"""
    dt, sp = (np.uint32, F32_SPECIALS) if width == 32 else (np.uint64, F64_SPECIALS)
    rng = np.random.default_rng(seed)
    out = rng.integers(0, np.iinfo(dt).max, n, dtype=dt, endpoint=True)
    pick = rng.random(n) < 0.7
    out[pick] = rng.choice(sp, int(pick.sum()))
    return out


def make(oracle, inp, n, width, seed):
    if inp == "L":
        return low_entropy(oracle, n, width, seed)
    if inp == "M":
        return mixed(n, width, seed)
    return floats(n, width, seed)


# ---- running one case -----------------------------------------------------------------------------------------------
def dev(a):
    return torch.from_numpy(a.view(np.int32 if a.dtype.itemsize == 4 else np.int64).copy()).cuda()


def host(t, dt):
    return t.cpu().numpy().view(dt)


def sort_and_compare(s, bits, order, *, kind="u", desc=False, begin=0, end=None, pairs=False, what=""):
    """Sort `bits` with the entry point the arguments name; keys (and payload = index) must equal the reference's."""
    width = bits.dtype.itemsize * 8
    tk = dev(bits)
    tv = torch.arange(bits.size, dtype=torch.int32, device="cuda") if pairs else None
    if end is not None:
        s.sort_bits(tk, begin, end, tv)
    elif kind != "u" or desc:
        name = f"{kind}{width}"
        if pairs:
            s.sort_pairs_typed(tk, tv, name, desc)
        else:
            s.sort_keys_typed(tk, name, desc)
    elif pairs:
        s.sort_pairs(tk, tv)
    else:
        s.sort_keys(tk)
    got = host(tk, bits.dtype)
    if not np.array_equal(got, bits[order]):
        j = int(np.nonzero(got != bits[order])[0][0])
        raise AssertionError(f"{what} keys differ from the stable sort first at index {j} of {bits.size}")
    if pairs:
        gv = host(tv, np.uint32)
        assert np.array_equal(gv, order.astype(np.uint32)), f"{what} payloads differ from the stable order"


def plan_of(s):
    return s.info("last_skip_mask"), s.info("last_hot_mask"), s.info("last_executed_passes")


def assert_plan(s, bits, kind="u", desc=False, begin=0, end=None, skip=True, hot=True, what=""):
    want = expected_plan(bits, kind, desc, begin, end, skip, hot)
    assert plan_of(s) == want, f"{what} plan (skip, hot, executed) {plan_of(s)}, expected {want}"
    return want


def atomic_rank_mode(s):
    """Pin the atomic rank mode: only there does the HOT kernel rank a tile's hot digit with one ballot per round and the
    other keys with the divergent atomic.  The default is not fixed -- osb200_create falls back to ballot ranking when
    its self-test of same-address atomic order fails -- and a case that silently ran in ballot mode would no longer test
    that path, so it skips and says why."""
    import gpusorting_b200 as g

    try:
        s.set_option("rank_mode", 0)
    except g.OneSweepError as e:
        if e.status != -3:  # OSB200_ERR_UNSUPPORTED: the self-test failed on this device
            raise
        pytest.skip("atomic ranking is unavailable here: the create-time self-test of same-address atomic order failed")
    assert s.info("rank_mode") == 0


@pytest.fixture(scope="module")
def g():
    import gpusorting_b200 as g

    return g


# ---- 1. HOT x typed keys ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("desc", [False, True])
@pytest.mark.parametrize("inp", ["L", "F"])
@pytest.mark.parametrize("kind", ["i", "f"])
def test_hot_typed_32(g, oracle, kind, inp, desc, n):
    """i32/f32 keys and pairs: the first executed pass encodes, the last decodes -- both of them HOT"""
    bits = make(oracle, inp, n, 32, 11 + n % 7)
    order = stable_order(bits, kind, desc)
    with g.OneSweepSorter(n, 4, 4) as s:
        atomic_rank_mode(s)
        for pairs in (False, True):
            sort_and_compare(s, bits, order, kind=kind, desc=desc, pairs=pairs, what=f"{kind}32 {inp} pairs={pairs}")
            _, hot, _ = assert_plan(s, bits, kind, desc)
            assert hot & 1 and hot & 8, "the encoding and the decoding pass must both be HOT"


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("desc", [False, True])
@pytest.mark.parametrize("kind,inp", [("i", "L"), ("f", "F")])
def test_hot_typed_64(g, oracle, kind, inp, desc, n):
    bits = make(oracle, inp, n, 64, 12)
    order = stable_order(bits, kind, desc)
    with g.OneSweepSorter(n, 8, 0) as s:
        atomic_rank_mode(s)
        sort_and_compare(s, bits, order, kind=kind, desc=desc, what=f"{kind}64 {inp}")
        _, hot, _ = assert_plan(s, bits, kind, desc)
        assert hot & 1 and (kind == "f" or hot & 0x80)


# ---- 2. HOT x skipping x typed keys (odd executed count: the copy-back runs) ------------------------------------------
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("desc", [False, True])
@pytest.mark.parametrize("negative", [False, True])
def test_hot_skip_typed_copy_back(g, negative, desc, n):
    """f32 keys of one sign whose low mantissa byte is zero: pass 0 is skipped (its encoded digit is the same for all),
    so pass 1 is the first EXECUTED pass -- HOT (40 % of the keys share byte 1) and the one that encodes.  Three passes
    execute: the result lands in the alt buffers and the copy-back moves keys and payloads home."""
    rng = np.random.default_rng(21 + negative * 2 + desc)
    bits = (rng.integers(0x3F0000, 0x470000, n).astype(np.uint32) << np.uint32(8))  # 0.5 .. 32768, low byte 0
    common = rng.random(n) < 0.4
    bits[common] = (bits[common] & np.uint32(0xFFFF00FF)) | np.uint32(0x5A00)
    if negative:
        bits |= np.uint32(0x80000000)
    order = stable_order(bits, "f", desc)
    with g.OneSweepSorter(n, 4, 4) as s:
        atomic_rank_mode(s)
        for pairs in (False, True):
            sort_and_compare(s, bits, order, kind="f", desc=desc, pairs=pairs, what=f"pairs={pairs}")
            skip, hot, executed = assert_plan(s, bits, "f", desc)
            assert skip == 0b0001 and executed == 3 and hot & 0b0010


# ---- 3. HOT x bit ranges --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("inp", ["L", "M"])
@pytest.mark.parametrize("begin,end", [(0, 29), (3, 14), (8, 32)])
def test_hot_bit_range_u32(g, oracle, begin, end, inp, n):
    """(0, 29): the last digit has 5 bits -> the few-bins scatter inside the HOT kernel; (3, 14): a 3-bit last digit at
    an unaligned shift; (8, 32): three passes, the copy-back runs"""
    bits = make(oracle, inp, n, 32, 31 + begin)
    order = stable_order(bits, begin=begin, end=end)
    with g.OneSweepSorter(n, 4, 4) as s:
        atomic_rank_mode(s)
        for pairs in (False, True):
            sort_and_compare(s, bits, order, begin=begin, end=end, pairs=pairs, what=f"[{begin},{end}) {inp} pairs={pairs}")
            _, hot, _ = assert_plan(s, bits, begin=begin, end=end)
            last = 1 << ((end - begin + 7) // 8 - 1)
            assert hot & last, "the narrow last digit must run in the HOT kernel"


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("inp", ["L", "M"])
@pytest.mark.parametrize("begin,end", [(17, 49), (0, 64)])
def test_hot_bit_range_u64(g, oracle, begin, end, inp, n):
    bits = make(oracle, inp, n, 64, 41 + begin)
    order = stable_order(bits, begin=begin, end=end)
    with g.OneSweepSorter(n, 8, 0) as s:
        atomic_rank_mode(s)
        sort_and_compare(s, bits, order, begin=begin, end=end, what=f"u64 [{begin},{end}) {inp}")
        _, hot, _ = assert_plan(s, bits, begin=begin, end=end)
        assert hot != 0


# ---- 4. HOT x forward-progress fallback -----------------------------------------------------------------------------
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("stall_every", [1, 3])
def test_hot_fallback_rereduces_stalled_tiles(g, oracle, stall_every, n):
    """Tiles withhold their reductions (test hook); the resident CTAs of the HOT kernel, striding over the tiles, must
    re-reduce them in the lookback -- from the encoded keys in the first pass of a typed sort."""
    bits = low_entropy(oracle, n, 32, 51)
    with g.OneSweepSorter(n, 4, 4) as s:
        atomic_rank_mode(s)
        s.set_option("spin_cap", 16)
        s.set_option("debug_stall_every", stall_every)
        order = stable_order(bits)
        for pairs in (False, True):
            sort_and_compare(s, bits, order, pairs=pairs, what=f"stall={stall_every} pairs={pairs}")
            assert assert_plan(s, bits)[1] == 0b1111
        order = stable_order(bits, "f", True)
        sort_and_compare(s, bits, order, kind="f", desc=True, what=f"f32 desc stall={stall_every}")
        assert assert_plan(s, bits, "f", True)[1] == 0b1111


# ---- 5. HOT x ballot ranking ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("inp", ["L", "M"])
def test_hot_ballot_rank_mode(g, oracle, inp, n):
    bits = make(oracle, inp, n, 32, 61)
    order = stable_order(bits)
    with g.OneSweepSorter(n, 4, 4) as s:
        s.set_option("rank_mode", 1)
        assert s.info("rank_mode") == 1
        for pairs in (False, True):
            sort_and_compare(s, bits, order, pairs=pairs, what=f"ballot {inp} pairs={pairs}")
            assert assert_plan(s, bits)[1] != 0
    b64 = make(oracle, inp, n, 64, 62)
    with g.OneSweepSorter(n, 8, 0) as s:
        s.set_option("rank_mode", 1)
        assert s.info("rank_mode") == 1
        sort_and_compare(s, b64, stable_order(b64), what=f"ballot u64 {inp}")
        assert assert_plan(s, b64)[1] != 0


# ---- 6. HOT tile variety --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", SIZES)
def test_hot_tile_variety(g, n):
    """The mixed input in the atomic rank mode: tiles whose hot digit is the pass's, one of their own, none (the
    per-tile rank falls back to the atomics), a tie, and the padding-dominated last tile"""
    bits = mixed(n, 32, 71)
    order = stable_order(bits)
    with g.OneSweepSorter(n, 4, 4) as s:
        atomic_rank_mode(s)
        for pairs in (False, True):
            sort_and_compare(s, bits, order, pairs=pairs, what=f"mixed pairs={pairs}")
            assert assert_plan(s, bits)[1] == 0b1111
    b64 = mixed(n, 64, 72)
    with g.OneSweepSorter(n, 8, 0) as s:
        atomic_rank_mode(s)
        sort_and_compare(s, b64, stable_order(b64), what="mixed u64")
        assert assert_plan(s, b64)[1] == 0xFF


# ---- 7. HOT == plain ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("inp", ["L", "M"])
def test_hot_and_plain_kernels_agree(g, oracle, inp, n):
    bits = make(oracle, inp, n, 32, 81)
    b64 = make(oracle, inp, n, 64, 82)
    outs = {}
    for hot in (1, 0):
        with g.OneSweepSorter(n, 4, 4) as s, g.OneSweepSorter(n, 8, 0) as s8:
            atomic_rank_mode(s)
            atomic_rank_mode(s8)
            s.set_option("hot_passes", hot)
            s8.set_option("hot_passes", hot)
            tk, tv = dev(bits), torch.arange(n, dtype=torch.int32, device="cuda")
            s.sort_pairs(tk, tv)
            assert_plan(s, bits, hot=bool(hot))
            t8 = dev(b64)
            s8.sort_keys(t8)
            assert_plan(s8, b64, hot=bool(hot))
            assert (s.info("last_hot_mask") != 0) == bool(hot) and (s8.info("last_hot_mask") != 0) == bool(hot)
            outs[hot] = (host(tk, np.uint32), host(tv, np.uint32), host(t8, np.uint64))
    for a, b in zip(outs[1], outs[0]):
        assert np.array_equal(a, b), "the HOT and the plain kernel disagree"
    order = stable_order(bits)
    assert np.array_equal(outs[0][0], bits[order]) and np.array_equal(outs[0][1], order.astype(np.uint32))
    assert np.array_equal(outs[0][2], np.sort(b64))


# ---- float specials below the HOT threshold -------------------------------------------------------------------------
@pytest.mark.parametrize("desc", [False, True])
@pytest.mark.parametrize("width", [32, 64])
@pytest.mark.parametrize("n", [5000, 300007])
def test_float_specials_total_order(g, width, desc, n):
    """NaNs of both signs and payloads, +-0, +-inf and denormals follow the IEEE total order of the bit patterns: -NaNs
    first, +NaNs last (reversed for descending, ties stable).  n = 5000 is the single-CTA small-n path, 300,007 the
    multi-kernel path."""
    bits = floats(n, width, 91 + width + desc)
    order = stable_order(bits, "f", desc)
    with g.OneSweepSorter(n, 4, 4) if width == 32 else g.OneSweepSorter(n, 8, 0) as s:
        assert (n <= s.info("small_path_max_n")) == (n == 5000)
        for pairs in (False, True) if width == 32 else (False,):
            sort_and_compare(s, bits, order, kind="f", desc=desc, pairs=pairs, what=f"f{width} pairs={pairs}")
    got = bits[order]
    fl = got.view(np.float32 if width == 32 else np.float64)
    neg = (got >> np.array(width - 1, dtype=got.dtype)).astype(bool)
    nan = np.isnan(fl)
    lo, hi = nan & neg, nan & ~neg  # -NaNs, +NaNs
    first, last = (lo, hi) if not desc else (hi, lo)
    k1, k2 = int(first.sum()), int(last.sum())
    assert k1 and k2 and first[:k1].all() and last[n - k2:].all()
    mid = fl[k1:n - k2]
    assert not np.isnan(mid).any() and (np.all(mid[1:] <= mid[:-1]) if desc else np.all(mid[1:] >= mid[:-1]))
    assert np.array_equal(radix_key(got, "f", desc), np.sort(radix_key(bits, "f", desc)))
