"""The certificates of tests/sortcheck.py on small CPU tensors: they accept the stable sort and reject every way of being
almost it.  No GPU needed; the GPU tests rely on these to be exact."""
import numpy as np
import pytest
import torch

from tests.sortcheck import (bincount_chunked, certify_sorted_multiset, certify_stable_sort, expected_plan, radix_key,
                             radix_key_torch, stable_order)

F32_SPECIALS = np.array([0x00000000, 0x80000000, 0x3F800000, 0xBF800000, 0x7F800000, 0xFF800000, 0x00000001, 0x807FFFFF,
                         0x7FC00000, 0x7FC00001, 0xFFC00000, 0xFFC12345, 0x7F800001, 0xFF800001], dtype=np.uint32)


def stable_sorted(bits, kind="u", desc=False, begin=0, end=None):
    order = stable_order(bits, kind, desc, begin, end)
    return bits[order], order


def tensors(bits, order=None):
    t = torch.from_numpy(bits.view(np.int32 if bits.dtype.itemsize == 4 else np.int64).copy())
    return t if order is None else (t, torch.from_numpy(order.astype(np.int64).astype(np.uint32).view(np.int32).copy()))


@pytest.mark.parametrize("kind", ["u", "i", "f"])
@pytest.mark.parametrize("desc", [False, True])
@pytest.mark.parametrize("width", [32, 64])
def test_radix_key_torch_matches_numpy(kind, desc, width):
    rng = np.random.default_rng(width * 7 + desc * 3 + ord(kind))
    dt = np.uint32 if width == 32 else np.uint64
    bits = rng.integers(0, np.iinfo(dt).max, 5000, dtype=dt, endpoint=True)
    bits[:4] = [0, np.iinfo(dt).max, np.iinfo(dt).max >> 1, (np.iinfo(dt).max >> 1) + 1]
    r = radix_key_torch(tensors(bits), kind, desc).numpy()
    want = radix_key(bits, kind, desc)
    # torch's signed order must be numpy's unsigned order
    assert np.array_equal(np.argsort(r, kind="stable"), np.argsort(want, kind="stable"))
    for begin, end in [(0, 8), (3, 14), (width - 5, width), (1, width)]:
        rb = radix_key_torch(tensors(bits), kind, desc, begin, end).numpy()
        field = (want >> dt(begin)) & dt((1 << (end - begin)) - 1)
        assert np.array_equal(rb, field.astype(np.int64)), (begin, end)


def test_radix_key_float_total_order():
    # -NaN < -inf < -1 < -denormal < -0 < +0 < +denormal < +1 < +inf < +NaN
    b = np.array([0x7FC00000, 0x3F800000, 0x00000001, 0x80000000, 0xFF800000, 0x00000000, 0xFFC00000, 0x7F800000,
                  0xBF800000, 0x807FFFFF], dtype=np.uint32)
    got = b[np.argsort(radix_key(b, "f"), kind="stable")]
    assert got.tolist() == [0xFFC00000, 0xFF800000, 0xBF800000, 0x807FFFFF, 0x80000000, 0x00000000, 0x00000001,
                            0x3F800000, 0x7F800000, 0x7FC00000]
    down = b[np.argsort(radix_key(b, "f", True), kind="stable")]
    assert down.tolist() == got.tolist()[::-1]


def test_expected_plan_models_skips_and_hot_places():
    n = 1 << 22
    k = np.full(n, 0x11223344, dtype=np.uint32)
    k[: n // 2] = 0x11220044  # byte 1 takes two values, half each: hot; the other bytes are constant: skipped
    assert expected_plan(k) == (0b1101, 0b0010, 1)
    assert expected_plan(k, skip=False) == (0, 0b1111, 4)
    assert expected_plan(k[:-1]) == (0b1101, 0, 1)  # below 2^22 nothing is hot
    assert expected_plan(k, begin=4, end=29) == (0b1100, 0b0011, 2)  # places at bits 4, 12, 20, 28 (1 bit)


@pytest.mark.parametrize("kind,desc", [("u", False), ("f", False), ("f", True), ("i", True)])
def test_certificate_accepts_the_stable_sort(kind, desc):
    rng = np.random.default_rng(1)
    bits = rng.choice(F32_SPECIALS, 3000) if kind == "f" else rng.integers(0, 40, 3000).astype(np.uint32)
    out, order = stable_sorted(bits, kind, desc)
    ik = tensors(bits)
    ok, ov = tensors(out, order)
    for chunk in (7, 64, 1 << 20):  # chunk boundaries inside runs of equal keys
        certify_stable_sort(ik, ok, ov, kind, desc, chunk=chunk)


def test_certificate_accepts_bit_range_and_u64_sorts():
    rng = np.random.default_rng(2)
    bits = rng.integers(0, 1 << 32, 2000, dtype=np.uint64).astype(np.uint32)
    out, order = stable_sorted(bits, begin=3, end=9)
    certify_stable_sort(tensors(bits), *tensors(out, order), begin=3, end=9, chunk=100)
    b64 = rng.integers(0, 8, 2000, dtype=np.uint64) << np.uint64(61)
    out, order = stable_sorted(b64)
    certify_stable_sort(tensors(b64), *tensors(out, order), chunk=333)


def corrupt(case, out, order, keys):
    out, order = out.copy(), order.copy()
    if case == "adjacent_inversion":  # two neighbours with different keys swapped (keys AND payloads: a consistent pair)
        j = int(np.nonzero(keys[1:] != keys[:-1])[0][0])
        out[[j, j + 1]] = out[[j + 1, j]]
        order[[j, j + 1]] = order[[j + 1, j]]
    elif case == "equal_keys_swapped":  # unstable: same keys, payloads out of input order
        j = int(np.nonzero(keys[1:] == keys[:-1])[0][0])
        order[[j, j + 1]] = order[[j + 1, j]]
    elif case == "duplicated_element":  # one element written twice, its neighbour lost
        j = int(np.nonzero(keys[1:] == keys[:-1])[0][0])
        order[j + 1] = order[j]
    elif case == "payload_mismatch":  # keys sorted, payload a permutation, but two payloads name each other's keys
        j = int(np.nonzero(keys[1:] != keys[:-1])[0][-1])
        order[[j, j + 1]] = order[[j + 1, j]]
    return out, order


@pytest.mark.parametrize("case", ["adjacent_inversion", "equal_keys_swapped", "duplicated_element", "payload_mismatch"])
@pytest.mark.parametrize("chunk", [5, 1 << 20])
def test_certificate_rejects_near_misses(case, chunk):
    rng = np.random.default_rng(3)
    bits = rng.integers(0, 16, 400).astype(np.uint32)
    out, order = stable_sorted(bits)
    bad_out, bad_order = corrupt(case, out, order, radix_key(out))
    with pytest.raises(AssertionError):
        certify_stable_sort(tensors(bits), *tensors(bad_out, bad_order), chunk=chunk)


def test_certificate_catches_an_inversion_across_a_chunk_boundary():
    bits = np.arange(100, dtype=np.uint32)
    out, order = bits.copy(), np.arange(100)
    out[[49, 50]], order[[49, 50]] = out[[50, 49]], order[[50, 49]]
    with pytest.raises(AssertionError, match="order"):
        certify_stable_sort(tensors(bits), *tensors(out, order), chunk=50)


def test_keys_only_certificate():
    C = 0x9E3779B1
    inv = pow(C, -1, 1 << 32)
    x = np.random.default_rng(4).integers(0, 1 << 10, 5000, dtype=np.uint64)
    keys = ((x * np.uint64(C)) & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    bin_of = lambda t: ((t.to(torch.int64) & 0xFFFFFFFF) * inv) & 0xFFFFFFFF  # noqa: E731  (the generator value back)
    counts = bincount_chunked(tensors(keys), bin_of, 1 << 10, chunk=999)
    good = np.sort(keys)
    certify_sorted_multiset(counts, tensors(good), bin_of, chunk=999)
    dup = good.copy()
    j = int(np.nonzero(good[1:] != good[:-1])[0][0])
    dup[j + 1] = dup[j]  # still sorted, one value lost and another doubled
    with pytest.raises(AssertionError, match="multiset"):
        certify_sorted_multiset(counts, tensors(dup), bin_of, chunk=999)
    swapped = good.copy()
    j = int(np.nonzero(good[998:] != good[997:-1])[0][0]) + 997  # an inversion at or after the first chunk boundary
    swapped[[j, j + 1]] = swapped[[j + 1, j]]
    with pytest.raises(AssertionError, match="order"):
        certify_sorted_multiset(counts, tensors(swapped), bin_of, chunk=999)
    alien = good.copy()
    alien[-1] = np.uint32(0xFFFFFFFF)  # a value outside the input's support (its bin is out of range)
    with pytest.raises(AssertionError, match="multiset"):
        certify_sorted_multiset(counts, tensors(alien), bin_of, chunk=999)
